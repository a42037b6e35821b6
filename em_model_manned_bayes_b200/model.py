"""Host-side mirror of the reference's model classes on top of the C ABI.

Mirrors (paths relative to /root/reference/code/matlab/):
  em_read.m                                  -> EncounterModel(parameters_filename=...)
  @EncounterModel/EncounterModel.m           -> EncounterModel properties (same names)
  bn_sample.m                                -> bn_sample(G, r, N, alpha, num_samples, start, order)
  @UncorEncounterModel/UncorEncounterModel.m -> UncorEncounterModel.sample(n_samples, sample_time, ...)
  @CorTerminalModel/sample.m                 -> CorTerminalModel.sample(nSamples, ...)

All sampling goes through libemb200.so (CUDA, sm_100a).  Nothing here computes samples on the CPU.
Values are 1-based (bins, variable ids) exactly as the MATLAB API returns them.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _lib as L


def _ptr(a):
    """numpy array / torch tensor / None -> void* (and keepalive)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


TRACK_TILE = 128   # tracks per tile of the dense layout (emb200.h: emb_track_out)


def untile(buf, nvar: int, n: int, T: int):
    """[ceil(T/4)][ceil(n/128)][nvar][128][4] -> (n, nvar, T).  Works on numpy arrays and torch tensors."""
    nch, ntile = (T + 3) // 4, (n + TRACK_TILE - 1) // TRACK_TILE
    a = buf.reshape(nch, ntile, nvar, TRACK_TILE, 4)
    a = a.transpose(1, 3, 2, 0, 4) if isinstance(a, np.ndarray) else a.permute(1, 3, 2, 0, 4)
    return a.reshape(ntile * TRACK_TILE, nvar, nch * 4)[:n, :, :T]


def tile(vals):
    """(n, nvar, T) -> the dense layout as a flat array (the inverse of `untile`; padding tracks and seconds are 0).  numpy in,
    numpy out; a torch tensor in, a tensor on its device out."""
    n, nvar, T = vals.shape
    nch, ntile = (T + 3) // 4, (n + TRACK_TILE - 1) // TRACK_TILE
    if not isinstance(vals, np.ndarray):
        pad = vals.new_zeros((ntile * TRACK_TILE, nvar, nch * 4))
        pad[:n, :, :T] = vals
        return pad.reshape(ntile, TRACK_TILE, nvar, nch, 4).permute(3, 0, 2, 1, 4).contiguous().reshape(-1)
    pad = np.zeros((ntile * TRACK_TILE, nvar, nch * 4), dtype=vals.dtype)
    pad[:n, :, :T] = vals
    return np.ascontiguousarray(pad.reshape(ntile, TRACK_TILE, nvar, nch, 4).transpose(3, 0, 2, 1, 4)).ravel()


def untile_bins(buf, n_dyn: int, n: int, T: int):
    return untile(buf, n_dyn, n, T)


def untile_values(buf, n_tv: int, n: int, T: int):
    return untile(buf, n_tv, n, T)


@dataclass
class TrackResult:
    """Compact result of `EncounterModel.sample_tracks` (one entry per track, global order)."""
    n: int
    T: int
    dyn_vars: List[int]            # 1-based ids of the dynamic variables (temporal_map(:,1))
    tv_vars: List[int]             # 1-based ids of the time-varying variables (dynamic or resampled)
    bins_tiled: Optional[object]
    values_tiled: Optional[object]
    init_bins: Optional[object]    # (n_initial, n) int8
    init_values: Optional[object]  # (n_initial, n) float64 == out_inits'
    attempts: Optional[object]

    @property
    def bins(self):
        """(n, n_dyn, T) int8 1-based bins; [:, d, c] is the bin during second c+1."""
        return untile_bins(self.bins_tiled, len(self.dyn_vars), self.n, self.T)

    @property
    def values(self):
        """(n, n_tv, T) float32 continuous values."""
        return untile_values(self.values_tiled, len(self.tv_vars), self.n, self.T)


class EncounterModel:
    """@EncounterModel/EncounterModel.m:75-153 (file-backed form) -- same property names.  `idxZeroBoundaries` defaults to
    empty like the class constructor's own inputParser (:87); `em_read` called directly defaults to [1 2 3] (em_read.m:34-40),
    which is what UncorEncounterModel below passes."""

    def __init__(self, parameters_filename: str = "", idxZeroBoundaries: Sequence[int] = (),
                 isOverwriteZeroBoundaries: bool = False, prior=0, _handle=None):
        self._h = C.c_void_p()
        lib = L.lib()
        if _handle is not None:
            self._h = _handle
        else:
            if not parameters_filename:
                raise L.EmbError(L.EMB_E_ARG, "parameters_filename is required")
            idx = (C.c_int32 * max(1, len(idxZeroBoundaries)))(*[int(v) for v in idxZeroBoundaries])
            L.check(lib.emb_model_load(str(parameters_filename).encode(), int(bool(isOverwriteZeroBoundaries)),
                                       idx, len(idxZeroBoundaries), C.byref(self._h)))
        self.parameters_filename = parameters_filename
        self._load_info()
        self.start = [None] * self.n_initial                 # EncounterModel.m:259-261
        self._prior = 0
        if prior != 0:
            self.prior = prior

    @classmethod
    def from_arrays(cls, G_initial, r_initial, N_initial, G_transition=None, r_transition=None, N_transition=None,
                    temporal_map=None, boundaries=None, resample_rates=None, dirichlet_initial=None,
                    dirichlet_transition=None):
        """The array form of the constructor (@EncounterModel/EncounterModel.m:106-114) over emb_model_from_arrays -- the
        call sequence of matlab/emb_handle.m: the tables handed over are the weights select_random.m:17 sums,
        N{i} + alpha{i}, so any prior (constant, 'dbe', stay, hand-made dirichlet cells) is reproduced exactly.
        N_* / dirichlet_*: one r_i x q_i array per variable (None for the first n_initial entries of the transition
        lists, like the reference's cells); G: [parent, child]."""
        def weights(N, alpha):
            out = []
            for i, t in enumerate(N or []):
                if t is None or np.size(t) == 0:
                    continue
                w = np.asarray(t, dtype=np.float64)
                if alpha is not None and alpha[i] is not None and np.size(alpha[i]):
                    w = w + np.asarray(alpha[i], dtype=np.float64)
                out.append(w.ravel(order="F"))
            return np.ascontiguousarray(np.concatenate(out)) if out else np.zeros(0)

        Gi = np.ascontiguousarray(np.asarray(G_initial, dtype=np.uint8))
        ri = np.ascontiguousarray(np.asarray(r_initial, dtype=np.int32).ravel())
        n = int(ri.size)
        wi = weights(N_initial, dirichlet_initial)
        nt = 0 if r_transition is None else int(np.size(r_transition))
        Gt = np.ascontiguousarray(np.asarray(G_transition, dtype=np.uint8)) if nt else None
        rt = np.ascontiguousarray(np.asarray(r_transition, dtype=np.int32).ravel()) if nt else None
        wt = weights(N_transition, dirichlet_transition) if nt else np.zeros(0)
        tm = np.ascontiguousarray(np.asarray(temporal_map if temporal_map is not None else np.zeros((0, 2)), dtype=np.int32).reshape(-1, 2))
        bl = [np.asarray(b, dtype=np.float64).ravel() for b in (boundaries if boundaries is not None else [[]] * n)]
        blen = np.ascontiguousarray(np.array([b.size for b in bl], dtype=np.int32))
        bflat = np.ascontiguousarray(np.concatenate(bl)) if sum(b.size for b in bl) else np.zeros(1)
        rates = np.ascontiguousarray(np.asarray(resample_rates if resample_rates is not None else np.zeros(n), dtype=np.float64).ravel())
        h = C.c_void_p()
        L.check(L.lib().emb_model_from_arrays(n, Gi.ctypes.data, ri.ctypes.data, wi.ctypes.data, wi.size, nt,
                                              Gt.ctypes.data if nt else None, rt.ctypes.data if nt else None,
                                              wt.ctypes.data if nt else None, wt.size, tm.ctypes.data, tm.shape[0],
                                              bflat.ctypes.data, blen.ctypes.data, rates.ctypes.data, C.byref(h)))
        self = cls.__new__(cls)
        EncounterModel.__init__(self, _handle=h)
        return self

    # -- lifetime ----------------------------------------------------------------------------------
    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                L.lib().emb_model_free(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    # -- properties --------------------------------------------------------------------------------
    def _load_info(self):
        lib = L.lib()
        info = L.ModelInfo()
        L.check(lib.emb_model_get_info(self._h, C.byref(info)))
        self._info = info
        n, nt = info.n_initial, info.n_transition
        self.n_initial, self.n_transition = n, nt
        self.n_dyn, self.n_gated, self.n_timevarying = info.n_dyn, info.n_gated, info.n_timevarying
        self.is_dynvar_depend = bool(info.is_dynvar_depend)
        self.r_initial = np.array(info.r_initial[:n], dtype=np.int64)
        self.r_transition = np.array(info.r_transition[:nt], dtype=np.int64)
        self.order_initial = list(info.order_initial[:n])
        self.order_transition = list(info.order_transition[:nt])
        self.temporal_map = np.array([[info.temporal_map[k][0], info.temporal_map[k][1]] for k in range(info.n_dyn)],
                                     dtype=np.int64).reshape(-1, 2)
        self.zero_bins = [[int(z)] if z else [] for z in info.zero_bins[:n]]
        self.resample_rates = np.array(info.resample_rates[:n], dtype=np.float64)
        self.bounds_initial = np.array([[info.bounds_initial[i][0], info.bounds_initial[i][1]] for i in range(n)])
        self.timevarying_vars = list(info.timevarying_vars[:info.n_timevarying])
        gv = (C.c_int32 * max(1, info.n_gated))()
        lib.emb_model_get_gated(self._h, gv, info.n_gated)
        self.gated_vars = list(gv[:info.n_gated])                # 1-based ids the packed event rows refer to by ordinal
        self.labels_initial = self._labels(0)
        self.labels_transition = self._labels(1) if nt else []
        G = np.zeros(n * n, dtype=np.uint8)
        lib.emb_model_get_G(self._h, 0, G.ctypes.data, G.size)
        self.G_initial = G.reshape(n, n).astype(bool)
        if nt:
            G = np.zeros(nt * nt, dtype=np.uint8)
            lib.emb_model_get_G(self._h, 1, G.ctypes.data, G.size)
            self.G_transition = G.reshape(nt, nt).astype(bool)
        else:
            self.G_transition = np.zeros((0, 0), dtype=bool)
        blen = list(info.boundaries_len[:n])
        flat = np.zeros(max(1, sum(blen)))
        lib.emb_model_get_boundaries(self._h, flat.ctypes.data, flat.size)
        self.boundaries, o = [], 0
        for k in blen:
            self.boundaries.append(flat[o:o + k].copy())
            o += k
        self.cutpoints_initial = [np.arange(2, self.r_initial[i] + 1, dtype=np.float64) if blen[i] == 0
                                  else self.boundaries[i][1:-1].copy() for i in range(n)]   # em_read.m:128-136

    def _labels(self, which):
        lib = L.lib()
        need = lib.emb_model_get_labels(self._h, which, None, 0)
        buf = C.create_string_buffer(int(need))
        lib.emb_model_get_labels(self._h, which, buf, need)
        s = buf.value.decode("utf-8")
        return s.split("\n") if s else []

    def _tables(self, which):
        lib = L.lib()
        total = int(self._info.len_N_transition if which else self._info.len_N_initial)
        flat = np.zeros(max(1, total))
        lib.emb_model_get_N(self._h, which, flat.ctypes.data, flat.size)
        G = self.G_transition if which else self.G_initial
        r = self.r_transition if which else self.r_initial
        nvar = G.shape[0]
        first = self.n_initial if which else 0
        out: List[Optional[np.ndarray]] = [None] * nvar
        o = 0
        for i in range(first, nvar):
            q = int(np.prod(r[G[:, i]])) if G[:, i].any() else 1
            cnt = int(r[i]) * q
            out[i] = flat[o:o + cnt].reshape((int(r[i]), q), order="F").copy()
            o += cnt
        return out

    @property
    def N_initial(self):
        return self._tables(0)

    @property
    def N_transition(self):
        return self._tables(1)

    @property
    def dediscretize_parameters(self):
        return self.boundaries

    @property
    def prior(self):
        return self._prior

    @prior.setter
    def prior(self, value):
        """EncounterModel.m:194-203: numeric constant or 'dbe' (bn_dirichlet_prior.m:17-38)."""
        lib = L.lib()
        if isinstance(value, str):
            if value.lower() != "dbe":
                raise L.EmbError(L.EMB_E_ARG, "prior:notdbe Unknown prior of %s, if char expecting prior = 'dbe'" % value)
            kind, v = L.EMB_PRIOR_DBE, 0.0
        else:
            kind, v = L.EMB_PRIOR_CONSTANT, float(value)
        L.check(lib.emb_set_prior(self._h, 0, kind, v))
        if self.n_transition:
            L.check(lib.emb_set_prior(self._h, 1, kind, v))
        self._prior = value

    def set_transition_stay_prior(self, value: float = 1.0):
        """setTransitionPriors.m:12-33 (terminal trajectory DBNs)."""
        L.check(L.lib().emb_set_prior(self._h, 1, L.EMB_PRIOR_STAY, float(value)))

    def packed(self, which: int) -> np.ndarray:
        lib = L.lib()
        n = lib.emb_model_get_packed(self._h, which, None, 0)
        buf = np.zeros(max(1, int(n)), dtype=np.uint32)
        lib.emb_model_get_packed(self._h, which, buf.ctypes.data, buf.size)
        return buf[:int(n)]

    # -- option plumbing ---------------------------------------------------------------------------
    def _opts(self, start=None, device=None, stream=None, mem=L.EMB_MEM_HOST, max_attempts=0, start_per_sample=None):
        """`start`: one preset per variable (the `start` cell of bn_sample.m:45; None / [] / NaN = free).
        `start_per_sample`: (n_samples, n_initial) presets, 0 / NaN = free -- the rows of
        @CorTerminalModel/InitStartTerminal.m, one per sample; a numpy array (host calls) or an int8 torch tensor of shape
        (n_initial, n_samples) already on the device the outputs live on."""
        o = L.SampleOpts()
        L.lib().emb_sample_opts_init(C.byref(o))
        if start_per_sample is not None:
            if isinstance(start_per_sample, np.ndarray) or isinstance(start_per_sample, (list, tuple)):
                a = np.nan_to_num(np.asarray(start_per_sample, dtype=np.float64), nan=0.0)
                if a.ndim != 2 or a.shape[1] != self.n_initial:
                    raise L.EmbError(L.EMB_E_ARG, "start_per_sample must be n_samples x n_initial")
                start_per_sample = np.ascontiguousarray(a.T.astype(np.int8))
            o._keep = start_per_sample                            # keep the buffer alive as long as the options
            o.start_per_sample = _ptr(start_per_sample)
            start = [None] * self.n_initial if start is None else start
        start = self.start if start is None else start
        if len(start) != self.n_initial:
            raise L.EmbError(L.EMB_E_ARG, "start must have n_initial entries")
        for i, s in enumerate(start):
            free = s is None or (isinstance(s, (list, tuple, np.ndarray)) and len(s) == 0) or \
                (isinstance(s, float) and math.isnan(s))
            o.start[i] = 0 if free else int(s)
        o.mem = mem
        o.device = -1 if device is None else int(device)
        o.stream = None if stream is None else int(stream)
        o.max_attempts = int(max_attempts)
        return o

    @staticmethod
    def _alloc(shape, dtype, like):
        """Allocate an output buffer: numpy (host) or torch on `like` device."""
        if like is None:
            return np.zeros(shape, dtype=dtype)
        import torch
        tdt = {np.int8: torch.int8, np.float32: torch.float32, np.float64: torch.float64, np.uint16: torch.int16, np.int16: torch.int16, np.uint8: torch.uint8,
               np.uint64: torch.int64, np.int64: torch.int64}[dtype]
        return torch.zeros(shape, dtype=tdt, device=like)

    @staticmethod
    def _empty_bytes(count, like):
        """An uninitialised uint8 buffer (text that a call overwrites): numpy, or torch on `like` device."""
        if like is None:
            return np.empty((count,), dtype=np.uint8)
        import torch
        return torch.empty((count,), dtype=torch.uint8, device=like)

    # -- sampling ----------------------------------------------------------------------------------
    def sample_initial(self, n: int, seed: int = 0, first_sample: int = 0, start=None, opts=None, device=None,
                       want_values=True, want_attempts=True, out=None, enqueue_only: bool = False, values_fp32: bool = False):
        """bn_sample.m:25-58 over n samples + de-discretisation.  Returns (bins (n, n_initial) int8,
        values (n, n_initial) float64 or None, attempts (n,) or None).  `device`: torch device string
        to keep the outputs in HBM; default host numpy."""
        o = opts if opts is not None else self._opts(start=start)
        stream = None
        if device is not None:
            import torch
            dev = torch.device(device)
            o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
            stream = torch.cuda.current_stream(dev).cuda_stream
            o.stream = stream
            if enqueue_only:      # EMB_MEM_ASYNC: queue the pass and return; async_status() collects the rejection flag
                o.mem |= L.EMB_MEM_ASYNC
        elif enqueue_only:
            raise L.EmbError(L.EMB_E_ARG, "enqueue_only needs device outputs")
        ni = self.n_initial
        if out is not None:       # reuse the buffers of a previous call: (bins.T, values.T, attempts) as returned
            bins, vals, att = out[0].T, (out[1].T if out[1] is not None else None), out[2]
        else:
            bins = self._alloc((ni, n), np.int8, device)
            vals = self._alloc((ni, n), np.float32 if values_fp32 else np.float64, device) if want_values else None
            att = self._alloc((n,), np.uint16, device) if want_attempts else None
        rng = L.Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_sample))
        fn = L.lib().emb_sample_initial_f32 if (values_fp32 and vals is not None) else L.lib().emb_sample_initial
        L.check(fn(self._h, C.byref(rng), n, C.byref(o), _ptr(bins), _ptr(vals), _ptr(att)))
        return bins.T, (vals.T if vals is not None else None), att

    def sample_tracks(self, n: int, T: int, seed: int = 0, first_sample: int = 0, start=None, opts=None, device=None,
                      want_bins=True, want_values=True, want_init=True, hist_initial=None, hist_transition=None,
                      out: Optional[TrackResult] = None, enqueue_only: bool = False) -> TrackResult:
        """Dense compact tracks (emb200.h: emb_sample_tracks).  `enqueue_only` (device outputs only): EMB_MEM_ASYNC, the pass
        is queued on the current stream and the call returns at once; `async_status()` later reports rejection exhaustion."""
        lib = L.lib()
        o = opts if opts is not None else self._opts(start=start)
        if enqueue_only and device is None:
            raise L.EmbError(L.EMB_E_ARG, "enqueue_only needs device outputs")
        if device is not None:
            import torch
            dev = torch.device(device)
            o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
            o.stream = torch.cuda.current_stream(dev).cuda_stream
            if enqueue_only:
                o.mem |= L.EMB_MEM_ASYNC
        ni = self.n_initial
        if out is None:
            nb = int(lib.emb_tracks_bins_len(self._h, n, T))
            nv = int(lib.emb_tracks_values_len(self._h, n, T))
            out = TrackResult(
                n=n, T=T, dyn_vars=[int(v) for v in self.temporal_map[:, 0]], tv_vars=list(self.timevarying_vars),
                bins_tiled=self._alloc((nb,), np.int8, device) if want_bins else None,
                values_tiled=self._alloc((nv,), np.float32, device) if want_values else None,
                init_bins=self._alloc((ni, n), np.int8, device) if want_init else None,
                init_values=self._alloc((ni, n), np.float64, device) if want_init else None,
                attempts=self._alloc((n,), np.uint16, device) if want_init else None)
        to = L.TrackOut(_ptr(out.bins_tiled), _ptr(out.values_tiled), _ptr(out.init_bins), _ptr(out.init_values),
                        _ptr(out.attempts), _ptr(hist_initial), _ptr(hist_transition))
        rng = L.Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_sample))
        L.check(lib.emb_sample_tracks(self._h, C.byref(rng), n, T, C.byref(o), C.byref(to)))
        return out

    # -- scoring (emb200.h: emb_loglik_initial / emb_loglik_tracks) ----------------------------------------------------
    def _score_call(self, arrays, device, correct_dbn):
        """Options and buffer kind of a scoring call: torch CUDA tensors in -> device buffers on their device, outputs as tensors;
        numpy in -> host buffers, computed on `device` (CUDA ordinal or torch device; default the current one)."""
        o = self._opts(start=[None] * self.n_initial)
        o.correct_dbn = int(bool(correct_dbn))
        like = None
        if not isinstance(arrays[0], np.ndarray):
            import torch
            dev = arrays[0].device
            if dev.type != "cuda" or any(a.device != dev for a in arrays):
                raise L.EmbError(L.EMB_E_ARG, "loglik: tensors must all be on one CUDA device (or pass numpy arrays)")
            o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
            o.stream = torch.cuda.current_stream(dev).cuda_stream
            like = dev
        elif device is not None:
            import torch
            dev = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
            o.device = dev.index if dev.index is not None else -1
        return o, like

    @staticmethod
    def _int8(a, like):
        if like is None:
            return np.ascontiguousarray(np.asarray(a), dtype=np.int8)
        import torch
        return a.to(torch.int8).contiguous()

    def loglik_initial(self, bins, device=None, per_var: bool = False):
        """log p(x) of initial-network bins under this model, sum_i log p(x_i | parents) in fp64 (emb_loglik_initial; the
        semantics are in include/emb200.h).  `bins`: (n, n_initial) 1-based, as `sample_initial` returns them.  numpy in, numpy
        out; a torch CUDA tensor in, tensors on its device out.  Returns total (n,) float64, and with `per_var` also the
        per-variable terms (n, n_initial): drop the columns of preset variables to get the conditional of the free ones."""
        o, like = self._score_call([bins], device, False)
        if bins.shape[1] != self.n_initial:
            raise L.EmbError(L.EMB_E_ARG, "loglik_initial: bins must be n x n_initial")
        b = self._int8(bins.T, like)                                       # the ABI's [n_initial][n]
        n = int(b.shape[1])
        total = self._alloc((n,), np.float64, like)
        pv = self._alloc((self.n_initial, n), np.float64, like) if per_var else None
        L.check(L.lib().emb_loglik_initial(self._h, n, _ptr(b), C.byref(o), _ptr(total), _ptr(pv)))
        return (total, pv.T) if per_var else total

    def loglik_tracks(self, init_bins, bins_tiled=None, T: Optional[int] = None, correct_dbn: bool = False, device=None):
        """log p of tracks under this model (emb_loglik_tracks): returns (initial (n,), transition (n,)) float64, the initial
        term scoring column 0 and the transition term summing columns 1..T-1 on the sampler's branch (frozen parents, or
        re-evaluated every second for models with a dynamic -> dynamic edge or with `correct_dbn`).
        `init_bins`: (n_initial, n) 1-based as `TrackResult.init_bins`, or a whole `TrackResult` (then `bins_tiled` and `T` come
        from it).  `bins_tiled`: the flat tiled layout of `sample_tracks`; turn plain (n, n_dyn, T) bins into it with `tile()`.
        numpy in, numpy out; torch CUDA tensors in, tensors on their device out."""
        if isinstance(init_bins, TrackResult):
            r = init_bins
            if r.init_bins is None or r.bins_tiled is None:
                raise L.EmbError(L.EMB_E_ARG, "loglik_tracks: the TrackResult needs init_bins and bins (want_init, want_bins)")
            init_bins, bins_tiled, T = r.init_bins, r.bins_tiled, r.T
        if bins_tiled is None or T is None:
            raise L.EmbError(L.EMB_E_ARG, "loglik_tracks: bins_tiled and T are required")
        o, like = self._score_call([init_bins, bins_tiled], device, correct_dbn)
        if init_bins.shape[0] != self.n_initial:
            raise L.EmbError(L.EMB_E_ARG, "loglik_tracks: init_bins must be n_initial x n")
        ib = self._int8(init_bins, like)
        n = int(ib.shape[1])
        bt = self._int8(bins_tiled, like).reshape(-1)
        if self.n_dyn and int(bt.shape[0]) != int(L.lib().emb_tracks_bins_len(self._h, n, int(T))):
            raise L.EmbError(L.EMB_E_ARG, "loglik_tracks: bins_tiled must have emb_tracks_bins_len(n, T) elements")
        init = self._alloc((n,), np.float64, like)
        trans = self._alloc((n,), np.float64, like)
        L.check(L.lib().emb_loglik_tracks(self._h, n, int(T), _ptr(ib), _ptr(bt), C.byref(o), _ptr(init), _ptr(trans)))
        return init, trans

    def loglik_events(self, events, offsets=None, T: Optional[int] = None, init_bins=None, dts=None, correct_dbn: bool = False,
                      device=None):
        """log p of tracks given as event lists (emb_loglik_track_events[_packed]): the same (initial (n,), transition (n,))
        float64 as `loglik_tracks` on the dense bins the lists expand to (`expand_events`), computed from the rows.
        `events`: a whole `EventResult` or `PackedEventResult` (it must carry init_bins), or raw rows -- emb_event rows
        (`EVENT_DTYPE` array, or the int64 tensor of a device `EventResult`), or packed words with their `dts` -- together
        with `offsets` (int64 [n+1]), `T` and `init_bins` (n_initial, n).  numpy in, numpy out; torch CUDA tensors in, tensors
        on their device out."""
        if isinstance(events, (EventResult, PackedEventResult)):
            r = events
            if r.init_bins is None:
                raise L.EmbError(L.EMB_E_ARG, "loglik_events: the result needs init_bins (want_init)")
            offsets, T, init_bins = r.offsets, r.T, r.init_bins
            events, dts = (r.words, r.dts) if isinstance(r, PackedEventResult) else (r.events, None)
        if offsets is None or T is None or init_bins is None:
            raise L.EmbError(L.EMB_E_ARG, "loglik_events: offsets, T and init_bins are required")
        arrays = [init_bins, events, offsets] + ([dts] if dts is not None else [])
        o, like = self._score_call(arrays, device, correct_dbn)
        if init_bins.shape[0] != self.n_initial:
            raise L.EmbError(L.EMB_E_ARG, "loglik_events: init_bins must be n_initial x n")
        ib = self._int8(init_bins, like)
        n = int(ib.shape[1])
        if like is None:
            off = np.ascontiguousarray(offsets, dtype=np.int64)
            ev = np.ascontiguousarray(events)
            dt = None if dts is None else np.ascontiguousarray(dts, dtype=np.uint8)
        else:
            off, ev, dt = offsets.contiguous(), events.contiguous(), None if dts is None else dts.contiguous()
        if int(off.shape[0]) != n + 1:
            raise L.EmbError(L.EMB_E_ARG, "loglik_events: offsets must have n + 1 entries")
        init = self._alloc((n,), np.float64, like)
        trans = self._alloc((n,), np.float64, like)
        lib = L.lib()
        if dt is None:
            rc = lib.emb_loglik_track_events(self._h, n, int(T), _ptr(ib), _ptr(ev), _ptr(off), C.byref(o), _ptr(init), _ptr(trans))
        else:
            rc = lib.emb_loglik_track_events_packed(self._h, n, int(T), _ptr(ib), _ptr(ev), _ptr(dt), _ptr(off), C.byref(o),
                                                    _ptr(init), _ptr(trans))
        L.check(rc)
        return init, trans

    # -- event lists -> out_samples and control rows (emb200.h: emb_track_events_expand[_packed]) ----------------------------
    def expand_events_gpu(self, events, offsets=None, T: Optional[int] = None, init_values=None, dts=None,
                          want_samples: bool = True, spec=None, device=None):
        """The other two outputs of UncorEncounterModel.sample, computed on the device from event lists.
        `events`: a whole `EventResult` or `PackedEventResult` (it must carry init_values), or raw rows -- emb_event rows
        (`EVENT_DTYPE` array, or the int64 tensor of a device `EventResult`), or packed words with their `dts` -- together
        with `offsets` (int64 [n+1]), `T` and `init_values` (n_initial, n) float64.
        `spec`: None for plain events2controls.m (the variables temporal_map(:,1), unscaled), or (vars, mul, div): 1-based
        initial variables and per column y = (x * mul) / div (`UncorEncounterModel.out_eme_spec()` gives the out_EME matrix).
        Returns (samples (n, T, n_initial) float64 or None -- samples[s] is out_samples{s}' -- and a `ControlsResult`).
        numpy in, numpy out; torch CUDA tensors in, tensors on their device out."""
        if isinstance(events, (EventResult, PackedEventResult)):
            r = events
            if r.init_values is None:
                raise L.EmbError(L.EMB_E_ARG, "expand_events_gpu: the result needs init_values (want_init)")
            offsets, T, init_values = r.offsets, r.T, r.init_values
            events, dts = (r.words, r.dts) if isinstance(r, PackedEventResult) else (r.events, None)
        if offsets is None or T is None or init_values is None:
            raise L.EmbError(L.EMB_E_ARG, "expand_events_gpu: offsets, T and init_values are required")
        arrays = [init_values, events, offsets] + ([dts] if dts is not None else [])
        o, like = self._score_call(arrays, device, False)
        if init_values.shape[0] != self.n_initial:
            raise L.EmbError(L.EMB_E_ARG, "expand_events_gpu: init_values must be n_initial x n")
        n, T = int(init_values.shape[1]), int(T)
        if like is None:
            iv = np.ascontiguousarray(init_values, dtype=np.float64)
            off = np.ascontiguousarray(offsets, dtype=np.int64)
            ev = np.ascontiguousarray(events)
            dt = None if dts is None else np.ascontiguousarray(dts, dtype=np.uint8)
        else:
            import torch
            iv, off, ev = init_values.to(torch.float64).contiguous(), offsets.contiguous(), events.contiguous()
            dt = None if dts is None else dts.contiguous()
        if int(off.shape[0]) != n + 1:
            raise L.EmbError(L.EMB_E_ARG, "expand_events_gpu: offsets must have n + 1 entries")
        cs = L.ControlsSpec()
        if spec is not None:
            vars_, mul, div = (list(c) for c in spec)
            if not (len(vars_) == len(mul) == len(div)) or len(vars_) > len(cs.vars):
                raise L.EmbError(L.EMB_E_ARG, "expand_events_gpu: spec needs equally long vars, mul and div of at most 8 columns")
            cs.n_cols = len(vars_)
            for j in range(cs.n_cols):
                cs.vars[j], cs.mul[j], cs.div[j] = int(vars_[j]), float(mul[j]), float(div[j])
        k = cs.n_cols or self.n_dyn
        samples = self._alloc((n, T, self.n_initial), np.float64, like) if want_samples else None
        ctl_off = self._alloc((n + 1,), np.int64, like)
        total = C.c_int64(0)
        lib = L.lib()

        def call(capacity, rows):
            if dt is None:
                return lib.emb_track_events_expand(self._h, n, T, _ptr(iv), _ptr(ev), _ptr(off), C.byref(o), C.byref(cs),
                                                   _ptr(samples), capacity, _ptr(rows), _ptr(ctl_off), C.byref(total))
            return lib.emb_track_events_expand_packed(self._h, n, T, _ptr(iv), _ptr(ev), _ptr(dt), _ptr(off), C.byref(o),
                                                      C.byref(cs), _ptr(samples), capacity, _ptr(rows), _ptr(ctl_off),
                                                      C.byref(total))

        rc = call(0, None)                                  # sizes the control rows (and writes everything if there are none)
        if rc == L.EMB_E_LIMIT and total.value > 0:
            rows = self._alloc((int(total.value), 1 + k), np.float64, like)
            rc = call(int(total.value), rows)
        else:
            rows = self._alloc((0, 1 + k), np.float64, like)
        L.check(rc)
        return samples, ControlsResult(rows=rows, offsets=ctl_off)

    # -- the text files of em_sample.m (emb200.h: emb_format_em_sample) --------------------------------------------------
    def format_em_sample(self, init_values=None, values_tiled=None, T: Optional[int] = None, first_id: int = 1,
                         n: Optional[int] = None, device=None):
        """initial.txt and transition.txt of em_sample.m without their header lines, formatted on the device exactly as
        printf's "%g" (and "%d" for the id of initial.txt) formats them.  `init_values`: (n_initial, n) float64, or a whole
        `TrackResult` (then `values_tiled`, `T` and `n` come from it); `values_tiled`: the flat dense tiles of `sample_tracks`
        for the same n and T.  A text whose input is None is skipped (then give `n`).  Track s has id first_id + s.
        Returns (initial, initial_offsets, transition, transition_offsets): uint8 text and int64 [n+1] offsets, None for a
        skipped text.  numpy in, numpy out (computed on `device`); torch CUDA tensors in, tensors on their device out."""
        if isinstance(init_values, TrackResult):
            r = init_values
            init_values, values_tiled, T, n = r.init_values, r.values_tiled, r.T, r.n
        if T is None or (init_values is None and (values_tiled is None or n is None)):
            raise L.EmbError(L.EMB_E_ARG, "format_em_sample: T, and init_values or n, are required")
        arrays = [a for a in (init_values, values_tiled) if a is not None]
        o, like = self._score_call(arrays, device, False)
        if init_values is not None:
            if init_values.shape[0] != self.n_initial:
                raise L.EmbError(L.EMB_E_ARG, "format_em_sample: init_values must be n_initial x n")
            n = int(init_values.shape[1])
        n, T = int(n), int(T)
        lib = L.lib()
        if like is None:
            iv = None if init_values is None else np.ascontiguousarray(init_values, dtype=np.float64)
            vt = None if values_tiled is None else np.ascontiguousarray(values_tiled, dtype=np.float32).reshape(-1)
        else:
            import torch
            iv = None if init_values is None else init_values.to(torch.float64).contiguous()
            vt = None if values_tiled is None else values_tiled.to(torch.float32).contiguous().reshape(-1)
        if vt is not None and int(vt.shape[0]) != int(lib.emb_tracks_values_len(self._h, n, T)):
            raise L.EmbError(L.EMB_E_ARG, "format_em_sample: values_tiled must have emb_tracks_values_len(n, T) elements")
        off = [self._alloc((n + 1,), np.int64, like) if a is not None else None for a in (iv, vt)]
        totals = (C.c_int64 * 2)()

        def call(caps, bufs):
            return lib.emb_format_em_sample(self._h, n, T, int(first_id), _ptr(iv), _ptr(vt), C.byref(o), caps[0], _ptr(bufs[0]),
                                            _ptr(off[0]), caps[1], _ptr(bufs[1]), _ptr(off[1]), totals)

        # One call into buffers of the longest possible text (emb_format.cuh: a "%g" has at most 13 bytes, an id's "%d" at
        # most 16 below 2^53), so the count pass runs once; the exact totals and a second call only if that bound were short.
        bound = [n * (17 + 14 * self.n_initial) if off[0] is not None else 0,
                 n * T * (28 + 14 * self.n_dyn) if off[1] is not None else 0]
        bufs = [self._empty_bytes(bound[f], like) if off[f] is not None else None for f in range(2)]
        rc = call(bound, bufs)
        if rc == L.EMB_E_LIMIT:
            bufs = [self._empty_bytes(int(totals[f]), like) if off[f] is not None else None for f in range(2)]
            rc = call((int(totals[0]), int(totals[1])), bufs)
        L.check(rc)
        bufs = [None if b is None else b[:int(totals[f])] for f, b in enumerate(bufs)]
        return bufs[0], off[0], bufs[1], off[1]


def async_status(device: int = -1) -> None:
    """Synchronise `device` and raise if an enqueue_only pass exhausted its rejection loop (emb_async_status)."""
    L.check(L.lib().emb_async_status(int(device)))


@dataclass
class EventResult:
    """Sparse result of `EncounterModel.sample_events`: row k of track s is events[offsets[s] + k]."""
    n: int
    T: int
    events: object        # structured array (host) or int64 tensor viewing emb_event rows (device)
    offsets: object       # int64 [n + 1]
    init_bins: Optional[object]
    init_values: Optional[object]
    attempts: Optional[object]
    total: int

    def track(self, s: int) -> np.ndarray:
        """out_events{s+1} as a k x 3 float64 matrix [dt, var, value] (host results only)."""
        o = np.asarray(self.offsets)
        e = np.asarray(self.events)[int(o[s]):int(o[s + 1])]
        return np.stack([e["dt"].astype(np.float64), e["var"].astype(np.float64), e["value"].astype(np.float64)], axis=1)


@dataclass
class PackedEventResult:
    """Result of `EncounterModel.sample_events_packed`: the 5-byte rows of emb_sample_track_events_packed.
    Row k of track s is (words[offsets[s] + k], dts[offsets[s] + k]); `decode()` gives the reference's [dt, var, value]."""
    n: int
    T: int
    words: object         # uint32 (host) / int32 tensor (device)
    dts: object           # uint8
    offsets: object       # int64 [n + 1]
    init_bins: Optional[object]
    init_values: Optional[object]
    attempts: Optional[object]
    total: int
    gated_vars: List[int]
    boundaries: List[np.ndarray]
    zero_bins: List[List[int]]

    def decode(self):
        """-> (dt int64, var int64 (1-based, 0 = closing row), bin int64 (1-based), value float64) over all rows.
        value = dediscretize.m:22-41 with u = (frac + 0.5) 2^-23, evaluated in fp64 on the host."""
        w = np.asarray(self.words.cpu() if hasattr(self.words, "cpu") else self.words).view(np.uint32).astype(np.int64)
        d = np.asarray(self.dts.cpu() if hasattr(self.dts, "cpu") else self.dts).astype(np.int64)
        gord = (w >> 27) & 7
        dt = d | ((w >> 30) << 8)
        b = ((w >> 23) & 15) + 1
        u = ((w & 0x7FFFFF).astype(np.float64) + 0.5) * 2.0 ** -23
        var = np.zeros_like(gord)
        val = np.zeros(len(w))
        binv = np.where(gord > 0, b, 0)
        for k, v in enumerate(self.gated_vars, start=1):
            m = gord == k
            if not m.any():
                continue
            var[m] = v
            e = np.asarray(self.boundaries[v - 1], dtype=np.float64)
            if e.size == 0:
                val[m] = b[m]                                          # dediscretize.m:7-10
                continue
            bb = b[m]
            x = e[bb - 1] + (e[bb] - e[bb - 1]) * u[m]                 # :39
            if self.zero_bins[v - 1]:
                x = np.where(bb == self.zero_bins[v - 1][0], 0.0, x)   # :24-25
            val[m] = x
        return dt, var, binv, val

    def track(self, s: int) -> np.ndarray:
        """out_events{s+1} as a k x 3 float64 matrix [dt, var, value]."""
        dt, var, _, val = self.decode()
        o = np.asarray(self.offsets.cpu() if hasattr(self.offsets, "cpu") else self.offsets)
        a, b = int(o[s]), int(o[s + 1])
        return np.stack([dt[a:b].astype(np.float64), var[a:b].astype(np.float64), val[a:b]], axis=1)


@dataclass
class ControlsResult:
    """Control rows of `EncounterModel.expand_events_gpu`: rows[offsets[s]:offsets[s+1]] belong to track s."""
    rows: object          # (total, 1 + k) float64: [t, y_1 .. y_k]
    offsets: object       # int64 [n + 1]

    def track(self, s: int):
        """the control matrix of track s (events2controls.m, or the out_EME event matrix with that spec)"""
        return self.rows[int(self.offsets[s]):int(self.offsets[s + 1])]


def _row_times(dt: np.ndarray, offsets: np.ndarray) -> np.ndarray:
    """Seconds elapsed at the END of every row's hold (dt summed from the first row of the row's own track)."""
    cum = np.cumsum(dt, dtype=np.int64)
    first = np.asarray(offsets[:-1], dtype=np.int64)
    before = np.where(first > 0, cum[np.maximum(first, 1) - 1], 0)          # total of the tracks before each track
    return cum - np.repeat(before, np.diff(np.asarray(offsets, dtype=np.int64)))


def expand_events(initial: np.ndarray, dt, var, value, offsets, T: int) -> np.ndarray:
    """Batch form of events2samples.m:9-27 for the rows of many tracks at once.

    initial (n, n_initial); dt / var / value: the rows of all tracks back to back; offsets int64 [n+1].
    -> (n, n_initial, T): column c is the state during second c+1.  A row [dt, var, value] lets the current state
    hold for dt more seconds and then sets `var`, so its value is visible from column sum(dt up to and including the
    row) on; of several rows that set the same variable in the same second the last one is the visible one.  Built
    without a per-row loop: the row that owns each (track, variable, column) is found by sorting, then carried forward
    in time with a running maximum of row ids."""
    initial = np.asarray(initial, dtype=np.float64)
    n, ni = initial.shape
    dt = np.asarray(dt, dtype=np.int64)
    var = np.asarray(var, dtype=np.int64)
    value = np.asarray(value, dtype=np.float64)
    offsets = np.asarray(offsets, dtype=np.int64)
    col = _row_times(dt, offsets)
    trk = np.repeat(np.arange(n, dtype=np.int64), np.diff(offsets))
    rows = np.nonzero((var > 0) & (col < T))[0]
    owner = np.full(n * ni * T, -1, dtype=np.int64)
    if rows.size:
        key = (trk[rows] * ni + (var[rows] - 1)) * T + col[rows]
        uniq, first_rev = np.unique(key[::-1], return_index=True)              # first in reversed order = last row of the key
        owner[uniq] = rows[::-1][first_rev]
    owner = np.maximum.accumulate(owner.reshape(n, ni, T), axis=2)
    return np.where(owner >= 0, value[np.maximum(owner, 0)], initial[:, :, None])


def controls_of(dense: np.ndarray, dt, offsets, var_cols: Sequence[int]) -> List[np.ndarray]:
    """Batch form of events2controls.m:9-31: for every row with dt > 0, [t, x(var_cols)] with t the second the hold starts
    and x the state during the hold -- read from the expanded matrix instead of replaying the list.
    -> one (k_i, 1 + len(var_cols)) matrix per track."""
    dt = np.asarray(dt, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    n = dense.shape[0]
    t0 = _row_times(dt, offsets) - dt
    trk = np.repeat(np.arange(n, dtype=np.int64), np.diff(offsets))
    keep = np.nonzero(dt > 0)[0]
    x = dense[trk[keep][:, None], np.asarray(var_cols, dtype=np.int64)[None, :], t0[keep][:, None]]
    ctl = np.concatenate([t0[keep][:, None].astype(np.float64), x], axis=1)
    cuts = np.searchsorted(keep, offsets[1:-1])
    return np.split(ctl, cuts)


def events2samples(initial, events) -> np.ndarray:
    """events2samples.m:9-27 for one track: (n_initial,) initial vector and k x 3 [dt var value] rows -> n_initial x T."""
    ev = np.asarray(events, dtype=np.float64).reshape(-1, 3)
    T = int(ev[:, 0].sum())
    return expand_events(np.asarray(initial, dtype=np.float64)[None, :], ev[:, 0], ev[:, 1], ev[:, 2],
                         np.array([0, ev.shape[0]]), T)[0]


def events2controls(initial, events, temporal_map) -> np.ndarray:
    """events2controls.m:9-31 for one track: one row [t, x(temporal_map(:,1))] per event with dt > 0."""
    ev = np.asarray(events, dtype=np.float64).reshape(-1, 3)
    off = np.array([0, ev.shape[0]])
    T = int(ev[:, 0].sum())
    dense = expand_events(np.asarray(initial, dtype=np.float64)[None, :], ev[:, 0], ev[:, 1], ev[:, 2], off, T)
    return controls_of(dense, ev[:, 0], off, np.asarray(temporal_map)[:, 0] - 1)[0]


class EncounterModelEvents:
    """@EncounterModelEvents/EncounterModelEvents.m:18-49: times at which the aircraft dynamics change.
    `event` is the k x 4 matrix [time_s, verticalRate_fps, turnRate_radps, longitudeAccel_ftpss] (at least one row)."""

    def __init__(self, event=None, time_s=0.0, verticalRate_fps=0.0, turnRate_radps=0.0, longitudeAccel_ftpss=0.0):
        if event is not None:
            self.event = event
        else:
            cols = [np.atleast_1d(np.asarray(c, dtype=np.float64)).ravel()
                    for c in (time_s, verticalRate_fps, turnRate_radps, longitudeAccel_ftpss)]
            if len({c.size for c in cols}) != 1:                                   # EncounterModelEvents.m:77
                raise L.EmbError(L.EMB_E_ARG, "Sizes of time_s, verticalRate_fps, turnRate_radps, longitudeAccel_ftpss are not equal")
            self.time_s, self.verticalRate_fps, self.turnRate_radps, self.longitudeAccel_ftpss = cols

    @property
    def event(self) -> np.ndarray:
        m = np.stack([self.time_s, self.verticalRate_fps, self.turnRate_radps, self.longitudeAccel_ftpss], axis=1)
        return m if m.shape[0] else np.zeros((1, 4))                              # :44-47

    @event.setter
    def event(self, m):
        m = np.asarray(m, dtype=np.float64)
        if m.ndim != 2 or m.shape[1] != 4:                                        # :35
            raise L.EmbError(L.EMB_E_ARG, "event matrix must have 4 columns")
        self.time_s, self.verticalRate_fps, self.turnRate_radps, self.longitudeAccel_ftpss = (m[:, k].copy() for k in range(4))


def _find(labels, name):
    for i, l in enumerate(labels):
        if l == name:
            return i + 1
    return 0


def _sample_events(self, n: int, T: int, seed: int = 0, first_sample: int = 0, start=None, opts=None, device=None,
                   want_init=True, capacity: Optional[int] = None) -> EventResult:
    """Sparse tracks (emb200.h: emb_sample_track_events): the reference's out_events lists."""
    lib = L.lib()
    o = opts if opts is not None else self._opts(start=start)
    if device is not None:
        import torch
        dev = torch.device(device)
        o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
        o.stream = torch.cuda.current_stream(dev).cuda_stream
    ni = self.n_initial
    ib = self._alloc((ni, n), np.int8, device) if want_init else None
    iv = self._alloc((ni, n), np.float64, device) if want_init else None
    att = self._alloc((n,), np.uint16, device) if want_init else None
    init = L.TrackOut(None, None, _ptr(ib), _ptr(iv), _ptr(att), None, None)
    rng = L.Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_sample))
    total = C.c_int64(0)
    if capacity is None:   # expected rows: T * (sum of rates + a transition allowance) + slack
        capacity = int(n * (T * (float(np.sum(self.resample_rates)) + 0.15) + 8)) + 1024

    def alloc(cap):
        if device is None:
            return np.zeros(max(cap, 1), dtype=L.EVENT_DTYPE), np.zeros(n + 1, dtype=np.int64)
        import torch
        return torch.zeros(max(cap, 1), dtype=torch.int64, device=device), torch.zeros(n + 1, dtype=torch.int64, device=device)

    ev, off = alloc(capacity)
    rc = lib.emb_sample_track_events(self._h, C.byref(rng), n, T, C.byref(o), capacity, _ptr(ev), _ptr(off), C.byref(init),
                                     C.byref(total))
    if rc == L.EMB_E_LIMIT and total.value > capacity:
        capacity = int(total.value)
        ev, off = alloc(capacity)
        rc = lib.emb_sample_track_events(self._h, C.byref(rng), n, T, C.byref(o), capacity, _ptr(ev), _ptr(off),
                                         C.byref(init), C.byref(total))
    L.check(rc)
    return EventResult(n=n, T=T, events=ev[:total.value], offsets=off, init_bins=ib, init_values=iv, attempts=att,
                       total=int(total.value))


EncounterModel.sample_events = _sample_events


def _sample_events_packed(self, n: int, T: int, seed: int = 0, first_sample: int = 0, start=None, opts=None, device=None,
                          want_init=True, capacity: Optional[int] = None) -> PackedEventResult:
    """Sparse tracks as 5-byte packed rows (emb200.h: emb_sample_track_events_packed): what crosses PCIe."""
    lib = L.lib()
    o = opts if opts is not None else self._opts(start=start)
    if device is not None:
        import torch
        dev = torch.device(device)
        o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
        o.stream = torch.cuda.current_stream(dev).cuda_stream
    ni = self.n_initial
    ib = self._alloc((ni, n), np.int8, device) if want_init else None
    iv = self._alloc((ni, n), np.float64, device) if want_init else None
    att = self._alloc((n,), np.uint16, device) if want_init else None
    init = L.TrackOut(None, None, _ptr(ib), _ptr(iv), _ptr(att), None, None)
    rng = L.Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_sample))
    total = C.c_int64(0)
    if capacity is None:
        capacity = int(n * (T * (float(np.sum(self.resample_rates)) + 0.15) + 8)) + 1024

    def alloc(cap):
        if device is None:
            return np.zeros(max(cap, 1), dtype=np.uint32), np.zeros(max(cap, 1), dtype=np.uint8), np.zeros(n + 1, dtype=np.int64)
        import torch
        return (torch.zeros(max(cap, 1), dtype=torch.int32, device=device), torch.zeros(max(cap, 1), dtype=torch.uint8, device=device),
                torch.zeros(n + 1, dtype=torch.int64, device=device))

    w, d, off = alloc(capacity)
    rc = lib.emb_sample_track_events_packed(self._h, C.byref(rng), n, T, C.byref(o), capacity, _ptr(w), _ptr(d), _ptr(off),
                                            C.byref(init), C.byref(total))
    if rc == L.EMB_E_LIMIT and total.value > capacity:
        capacity = int(total.value)
        w, d, off = alloc(capacity)
        rc = lib.emb_sample_track_events_packed(self._h, C.byref(rng), n, T, C.byref(o), capacity, _ptr(w), _ptr(d), _ptr(off),
                                                C.byref(init), C.byref(total))
    L.check(rc)
    return PackedEventResult(n=n, T=T, words=w[:total.value], dts=d[:total.value], offsets=off, init_bins=ib, init_values=iv,
                             attempts=att, total=int(total.value), gated_vars=list(self.gated_vars),
                             boundaries=self.boundaries, zero_bins=self.zero_bins)


EncounterModel.sample_events_packed = _sample_events_packed


class UncorEncounterModel(EncounterModel):
    """@UncorEncounterModel/UncorEncounterModel.m (file input_type)."""

    def __init__(self, parameters_filename: str, idxZeroBoundaries: Sequence[int] = (1, 2, 3),
                 isOverwriteZeroBoundaries: bool = False, prior=0):
        super().__init__(parameters_filename, idxZeroBoundaries, isOverwriteZeroBoundaries, prior)
        self.isRotorcraft = "rotorcraft" in str(parameters_filename)          # UncorEncounterModel.m:179-183
        self.idxL = _find(self.labels_initial, '"L"')                          # :225-229
        self.idxV = _find(self.labels_initial, '"v"')
        self.idxDV = _find(self.labels_initial, '"\\dot v"')
        self.idxDH = _find(self.labels_initial, '"\\dot h"')
        self.idxDPsi = _find(self.labels_initial, '"\\dot \\psi"')

    def uncor_opts(self, isQuantize500=False, layers=None, start=None, max_attempts=0, correct_dbn=False):
        if not (self.idxDV and self.idxDH and self.idxDPsi):                   # :231-234
            raise L.EmbError(L.EMB_E_ARG, "dynvar:empty Model does not have a dynamic variable for either "
                             "acceleration, vertical rate, or turn rate")
        o = self._opts(start=start, max_attempts=max_attempts)
        o.reject_mode = L.EMB_REJECT_UNCOR
        o.idx_v, o.idx_dh, o.idx_L = self.idxV, self.idxDH, self.idxL
        o.is_quantize500 = int(bool(isQuantize500))
        o.correct_dbn = int(bool(correct_dbn))       # not the reference's behaviour: parents re-evaluated every second
        if layers is not None and len(layers):
            layers = np.asarray(layers, dtype=np.float64).reshape(-1, 2)
            o.n_layers = layers.shape[0]
            for k in range(layers.shape[0]):
                o.layers[k][0], o.layers[k][1] = layers[k, 0], layers[k, 1]
        return o

    def sample_compact(self, n_samples: int, sample_time: int, seed: int = 0, first_sample: int = 0,
                       isQuantize500=False, layers=None, device=None, **kw) -> TrackResult:
        """The batch form of UncorEncounterModel.m:244-307 with compact dense outputs."""
        o = self.uncor_opts(isQuantize500, layers)
        return self.sample_tracks(n_samples, sample_time, seed=seed, first_sample=first_sample, opts=o,
                                  device=device, **kw)

    def sample_events_uncor(self, n_samples: int, sample_time: int, seed: int = 0, first_sample: int = 0,
                            isQuantize500=False, layers=None, device=None, **kw) -> EventResult:
        """The batch form of UncorEncounterModel.m:244-307 with the reference's sparse outputs."""
        return self.sample_events(n_samples, sample_time, seed=seed, first_sample=first_sample,
                                  opts=self.uncor_opts(isQuantize500, layers), device=device, **kw)

    def getDynamicLimits(self, initial, results=None, idx_G=None, idx_A=None, idx_L=None, idx_V=None, idx_DH=None,
                         is_discretized=None):
        """@UncorEncounterModel/getDynamicLimits.m:1-129: speed and vertical-rate limits from the 1st/99th percentiles of
        the count tables, conditioned on (G, A, L, v) when the model has them in positions 1, 2, 3, 4, 6 (:16).
        `initial`: 1 x n_initial values (bins where is_discretized[i], continuous otherwise); `results`: dict with
        `up_ft` and `speed_ftps` (only read for non-discretised L / v, :35-56).  Host-side table arithmetic."""
        def disc(x, cut):                                    # discretize_bayes.m:14-22
            x = np.atleast_1d(np.asarray(x, dtype=np.float64))
            cut = np.asarray(cut, dtype=np.float64)
            return np.array([cut.size + 1 if v >= cut[-1] else int(np.nonzero(v < cut)[0][0]) + 1 for v in x])

        lab = self.labels_initial
        idx_G = _find(lab, '"G"') if idx_G is None else idx_G
        idx_A = _find(lab, '"A"') if idx_A is None else idx_A
        idx_L = self.idxL if idx_L is None else idx_L
        idx_V = self.idxV if idx_V is None else idx_V
        idx_DH = self.idxDH if idx_DH is None else idx_DH
        if is_discretized is None:
            is_discretized = [len(b) == 0 for b in self.boundaries]
        N, r = self.N_initial, self.r_initial
        if all((idx_G, idx_A, idx_L, idx_V, idx_DH)) and (idx_G, idx_A, idx_L, idx_V, idx_DH) == (1, 2, 3, 4, 6):   # :16
            initial = np.asarray(initial, dtype=np.float64)
            one = lambda i: int(initial[i - 1]) if is_discretized[i - 1] else int(disc(initial[i - 1], self.cutpoints_initial[i - 1])[0])
            dG, dA = one(idx_G), one(idx_A)                                                            # :19-30
            if is_discretized[idx_L - 1]:
                dL = [int(initial[idx_L - 1])]
            else:                                                                                      # :35-38
                d = disc([np.min(results["up_ft"]), np.max(results["up_ft"])], self.cutpoints_initial[idx_L - 1])
                dL = list(range(int(d.min()), int(d.max()) + 1))
            if is_discretized[idx_V - 1]:
                dV = [int(initial[idx_V - 1])]
            else:                                                                                      # :46-50
                kts = np.asarray(results["speed_ftps"], dtype=np.float64) * 0.592484
                d = disc([kts.min(), kts.max()], self.cutpoints_initial[idx_V - 1])
                dV = list(range(int(d.min()), int(d.max()) + 1))
            rG, rA, rL, rV = int(r[idx_G - 1]), int(r[idx_A - 1]), int(r[idx_L - 1]), int(r[idx_V - 1])
            v_G = N[idx_V - 1][:, dG - 1::rG]                                                          # :57-58
            dh_G = N[idx_DH - 1][:, dG - 1::rG]
            v_GA = v_G[:, dA - 1::rA]                                                                  # :61-62
            dh_GA = dh_G[:, dA - 1::rA]
            uL = sorted(set(dL))
            v_GAL = v_GA[:, [k - 1 for k in uL]]                                                       # :66
            dh_GAL = sum(dh_GA[:, k - 1::rL] for k in uL)                                              # :69-72
            dh_GALV = sum(dh_GAL[:, k - 1::rV] for k in sorted(set(dV)))                               # :75-78
            v_initial = v_GAL.sum(axis=1)
            dh_initial = dh_GALV.sum(axis=1)
        else:                                                                                          # :85-86
            v_initial = N[idx_V - 1].sum(axis=1)
            dh_initial = N[idx_DH - 1].sum(axis=1)

        def pct(w):                                                                                    # :93-96, :115-118
            cs = np.cumsum(100.0 * w / w.sum())
            return int(np.nonzero(cs >= 1)[0][0]) + 1, int(np.nonzero(cs >= 99)[0][0]) + 1

        k_lo, k_hi = pct(v_initial)
        bV = self.boundaries[idx_V - 1]
        min_speed, max_speed = bV[k_lo] * 1.68780972222222, bV[k_hi] * 1.68780972222222               # :99-100 (edge k+1, 1-based)
        if self.isRotorcraft and max_speed > 304:                                                      # :104-109
            max_speed = 304.0
        if (not self.isRotorcraft) and min_speed < 30:
            min_speed = 30.0
        k_lo, k_hi = pct(dh_initial)
        bH = self.boundaries[idx_DH - 1]
        vr = float(np.max(np.abs(np.array([bH[k_lo], bH[k_hi]]) / 60.0)))                              # :120
        if math.isnan(vr):
            vr = 0.0
        return dict(minVel_ft_s=float(min_speed), maxVel_ft_s=float(max_speed), maxVertRate_ft_s=vr)

    def out_eme_spec(self):
        """The control columns of out_EME (UncorEncounterModel.m:286-297): [dh ft/min -> ft/s, dpsi deg/s -> rad/s,
        dv kt/s -> ft/s^2] as (vars, mul, div) for `expand_events_gpu`: x / 60, (pi/180) * x, x * 1.68780972222222."""
        return [self.idxDH, self.idxDPsi, self.idxDV], [1.0, math.pi / 180.0, 1.68780972222222], [60.0, 1.0, 1.0]

    def sample_batch(self, n_samples: int, sample_time: int, seed=float("nan"), isQuantize500=False, layers=None, device=None,
                     packed: bool = True, want_samples: bool = False):
        """The four outputs of UncorEncounterModel.m:192-313 in batch form, all computed on the device:
        (out_inits (n, n_initial) float64, the event result (`PackedEventResult`, or with packed=False the 8-byte
        `EventResult` that `sample` reads), samples (n, sample_time, n_initial) float64 or None -- samples[s] is
        out_samples{s}' -- and the out_EME event matrices as a `ControlsResult`).  With packed=False the values are the
        fp32 row values `sample` reads, so samples and controls equal its out_samples and out_EME.event bit for bit.
        `device`: keep everything in HBM as torch tensors; default host numpy."""
        if isinstance(seed, float) and math.isnan(seed):
            seed = int(np.random.SeedSequence().generate_state(2, dtype=np.uint32).view(np.uint64)[0])
        o = self.uncor_opts(isQuantize500, layers)
        fn = self.sample_events_packed if packed else self.sample_events
        res = fn(n_samples, sample_time, seed=int(seed), opts=o, device=device)
        samples, ctl = self.expand_events_gpu(res, want_samples=want_samples, spec=self.out_eme_spec())
        out_inits = np.ascontiguousarray(res.init_values.T) if device is None else res.init_values.T
        return out_inits, res, samples, ctl

    def sample(self, n_samples: int, sample_time: int, seed=float("nan"), isQuantize500=False, layers=None):
        """UncorEncounterModel.m:192-313 -> (out_inits n x n_initial, out_events list of k x 3 [dt var value],
        out_samples list of n_initial x T, out_EME list of EncounterModelEvents whose `event` is [t, dh ft/s, dpsi rad/s, dv ft/s^2]).
        `seed` NaN draws a fresh 64-bit seed (the reference keeps the global stream; here streams are keyed).
        out_samples and the controls are expanded on the host from the event lists (expand_events / controls_of)."""
        if isinstance(seed, float) and math.isnan(seed):
            seed = int(np.random.SeedSequence().generate_state(2, dtype=np.uint32).view(np.uint64)[0])
        res = self.sample_events_uncor(n_samples, sample_time, seed=int(seed), isQuantize500=isQuantize500, layers=layers)
        out_inits = np.ascontiguousarray(res.init_values.T)
        ev, off = np.asarray(res.events), np.asarray(res.offsets, dtype=np.int64)
        dense = expand_events(out_inits, ev["dt"], ev["var"], ev["value"], off, sample_time)          # :283
        dyn = list(self.temporal_map[:, 0])
        ctl = controls_of(dense, ev["dt"], off, [v - 1 for v in (self.idxDH, self.idxDPsi, self.idxDV)])   # :286-292
        assert all(v in dyn for v in (self.idxDH, self.idxDPsi, self.idxDV))
        for c in ctl:
            c[:, 1] /= 60.0                       # :295 dh: ft/min -> ft/s
            c[:, 2] *= math.pi / 180.0            # :296 dpsi: deg2rad
            c[:, 3] *= 1.68780972222222           # :297 dv: kt/s -> ft/s^2
        out_events = [res.track(k) for k in range(n_samples)]
        out_samples = [dense[k] for k in range(n_samples)]
        out_EME = [EncounterModelEvents(event=c) for c in ctl]                                # :300
        return out_inits, out_events, out_samples, out_EME


@dataclass
class TrajectoryResult:
    """Batch result of `CorTerminalModel.create_encounters` (emb200.h: emb_traj_out)."""
    n: int
    tmax: int
    traj: object           # (5, 2, 2*tmax+1, n) float32: field, aircraft, slot (t_s = slot - tmax), encounter; NaN = no state
    len: object            # (4, n) int16: states of chain 2*aircraft + (0 forward, 1 backward)

    def encounter(self, s: int):
        """traj(1:2) of createEncounter.m:10,74-84 for encounter s: two dicts of float64 row vectors
        t_s, x_nm, y_nm, z_ft, heading_deg, v_ft_s (already concatenated and ordered in time)."""
        ln = np.asarray(self.len.cpu() if hasattr(self.len, "cpu") else self.len)[:, s]
        col = self.traj[:, :, :, s]
        col = np.asarray(col.cpu() if hasattr(col, "cpu") else col, dtype=np.float64)
        out = []
        for ac in range(2):
            lo, hi = self.tmax - (int(ln[2 * ac + 1]) - 1), self.tmax + int(ln[2 * ac]) - 1
            d = {"t_s": np.arange(lo - self.tmax, hi - self.tmax + 1, dtype=np.float64)}
            for f, name in enumerate(L.TRAJ_FIELDS):
                d[name] = col[f, ac, lo:hi + 1].copy()
            out.append(d)
        return out


class CorTerminalModel(EncounterModel):
    """@CorTerminalModel/CorTerminalModel.m + sample.m + createEncounter.m.

    The encounter *geometry* model is the object itself (CorTerminalModel.m:80).  The ten trajectory DBNs
    (mdlFwd1_1 ... mdlBck2_3, CorTerminalModel.m:12-30,86-100) are loaded with `load_trajectory_models`; their
    files are missing from the public checkout (SURVEY.md F5), so tests and bench use models of the same layout
    written by `synthetic.write_terminal_model_set`."""

    # @CorTerminalModel/getDynamicLimits.m:14-62 (minVel_ft_s, maxVel_ft_s)
    DYN_LIMITS = {"GENERIC": (50.0, 506.0), "RTCA228_A1": (169.0, 491.0), "RTCA228_A2": (68.0, 338.0),
                  "RTCA228_A3": (68.0, 186.0), "TEST": (68.0, 186.0)}
    # CorTerminalModel.m:62 file-name stems -> (aircraft, direction, intent)
    TRAJECTORY_SLOTS = (("ownship_landing_model", "own_fwd", 0), ("ownship_takeoff_model", "own_fwd", 1),
                        ("ownship_landing_model_reverse", "own_bck", 0), ("ownship_takeoff_model_reverse", "own_bck", 1),
                        ("intruder_landing_model", "int_fwd", 0), ("intruder_takeoff_model", "int_fwd", 1),
                        ("intruder_transit_model", "int_fwd", 2), ("intruder_landing_model_reverse", "int_bck", 0),
                        ("intruder_takeoff_model_reverse", "int_bck", 1), ("intruder_transit_model_reverse", "int_bck", 2))
    GEO_FIELDS = ("own_intent", "own_distance", "own_bearing", "own_alt", "own_heading", "own_speed",
                  "int_intent", "int_distance", "int_bearing", "int_alt", "int_heading", "int_speed")

    def __init__(self, parameters_filename: str, acType1: str = "GENERIC", acType2: str = "GENERIC",
                 parameters_directory: Optional[str] = None):
        super().__init__(parameters_filename)
        self.acType1, self.acType2 = acType1, acType2
        self.bounds_sample = np.stack([np.full(self.n_initial, -np.inf), np.full(self.n_initial, np.inf)], axis=1)
        self.idx_own_speed = _find(self.labels_initial, '"own_speed"')
        self.idx_int_speed = _find(self.labels_initial, '"int_speed"')
        self.trajectory_models = {}
        if parameters_directory is not None:
            self.load_trajectory_models(parameters_directory)

    def InitStartTerminal(self, nSamples: int = 1000000, airspace_class=(False, True, True, True), own_intent=(True, True),
                          int_intent=(True, True, True), isVerbose: bool = False):
        """@CorTerminalModel/InitStartTerminal.m:43-92: the `start` rows for every kept combination of airspace class x
        ownship intent x intruder intent, ceil(nSamples / n_combs) rows each, class slowest and intruder intent fastest.
        -> list of rows, each a list of n_initial entries (the preset bin for variables 1..3, None elsewhere); like the
        reference's cell it has n_combs * ceil(nSamples / n_combs) rows (>= nSamples)."""
        lab = self.labels_initial
        if lab[:3] != ['"airspace_class"', '"own_intent"', '"int_intent"']:                          # :31-33
            raise L.EmbError(L.EMB_E_ARG, "InitStartTerminal: the first three variables must be airspace_class, own_intent, int_intent")
        keep = [np.nonzero(np.asarray(k, dtype=bool))[0] + 1 for k in (airspace_class, own_intent, int_intent)]
        for k, sel in enumerate((airspace_class, own_intent, int_intent)):                           # :36-38
            if len(sel) != int(self.r_initial[k]):
                raise L.EmbError(L.EMB_E_ARG, "InitStartTerminal: one flag per bin of variable %d" % (k + 1))
        n_combs = len(keep[0]) * len(keep[1]) * len(keep[2])                                          # :47
        n_samples = max(int(nSamples), n_combs)                                                      # :50-53
        per = -(-n_samples // n_combs)                                                               # :56
        rows = []
        for ii in keep[0]:                                                                           # :67-90
            for jj in keep[1]:
                for kk in keep[2]:
                    if isVerbose:
                        print("encounters %d-%d, airspace_class = %d, own_intent = %d, int_intent = %d"
                              % (len(rows) + 1, len(rows) + per, ii, jj, kk))
                    rows += [[int(ii), int(jj), int(kk)] + [None] * (self.n_initial - 3) for _ in range(per)]
        return rows

    def _terminal_opts(self, start=None, max_attempts=0, start_per_sample=None):
        o = self._opts(start=start, max_attempts=max_attempts, start_per_sample=start_per_sample)
        o.reject_mode = L.EMB_REJECT_BOX
        lo, hi = self.bounds_sample[:, 0].copy(), self.bounds_sample[:, 1].copy()
        for idx, ac in ((self.idx_own_speed, self.acType1), (self.idx_int_speed, self.acType2)):   # sample.m:64-65
            if idx:
                vmin, vmax = self.DYN_LIMITS[ac.upper()]
                lo[idx - 1], hi[idx - 1] = max(lo[idx - 1], vmin), min(hi[idx - 1], vmax)
        for i in range(self.n_initial):
            o.box_lo[i], o.box_hi[i] = lo[i], hi[i]
        return o

    def sample_raw(self, nSamples: int, seed: int = 0, first_sample: int = 0, device=None, start_per_sample=None):
        """-> (outInits (n, 15) float64, bins (n, 15) int8, attempts).  `start_per_sample`: one `start` row per sample
        (e.g. the rows of InitStartTerminal; None entries = free) -- the whole batch in one call."""
        sps = None
        if start_per_sample is not None:
            sps = np.array([[0 if (v is None or (isinstance(v, float) and math.isnan(v))) else int(v) for v in row]
                            for row in start_per_sample], dtype=np.float64)
            if sps.shape[0] != nSamples:
                raise L.EmbError(L.EMB_E_ARG, "start_per_sample needs one row per sample")
            if device is not None:
                import torch
                sps = torch.from_numpy(np.ascontiguousarray(sps.T.astype(np.int8))).to(device)
        bins, vals, att = self.sample_initial(nSamples, seed=seed, first_sample=first_sample,
                                              opts=self._terminal_opts(start_per_sample=sps), device=device)
        return vals, bins, att

    def sample(self, nSamples: int, seed=float("nan")):
        """@CorTerminalModel/sample.m:1-82 -> (outInits, outSamples list of dict(field -> value))."""
        if isinstance(seed, float) and math.isnan(seed):
            seed = int(np.random.SeedSequence().generate_state(2, dtype=np.uint32).view(np.uint64)[0])
        out_inits, _, _ = self.sample_raw(nSamples, seed=int(seed))
        names = [l.replace('"', "") for l in self.labels_initial]                                   # sample.m:59
        out_samples = [dict(zip(names, row)) for row in out_inits]
        return out_inits, out_samples

    # -- trajectory DBNs -----------------------------------------------------------------------------
    def load_trajectory_models(self, parameters_directory: str, reference_reverse_quirk: bool = False):
        """CorTerminalModel.m:56-100: finds `*_<stem>.txt` for the ten trajectory models in the directory and applies
        the stay prior of createEncounter.m:129.  `reference_reverse_quirk=True` reproduces CorTerminalModel.m:97,100,
        where mdlBck2_2 and mdlBck2_3 both load the intruder *landing* reverse model (SURVEY.md F8)."""
        import glob
        loaded = {}
        for stem, group, k in self.TRAJECTORY_SLOTS:
            use = stem
            if reference_reverse_quirk and group == "int_bck":
                use = "intruder_landing_model_reverse"
            hits = sorted(glob.glob(os.path.join(parameters_directory, "*_" + use + ".txt")))
            if not hits:
                raise L.EmbError(L.EMB_E_IO, "trajectory model *_%s.txt not found in %s" % (use, parameters_directory))
            if hits[0] not in loaded:
                m = EncounterModel(hits[0])
                m.set_transition_stay_prior(1.0)
                loaded[hits[0]] = m
            self.trajectory_models[(group, k)] = loaded[hits[0]]
        return self

    def set_trajectory_models(self, models: dict):
        """models[(group, intent-1)] -> EncounterModel, group in own_fwd/own_bck/int_fwd/int_bck."""
        for m in set(models.values()):
            m.set_transition_stay_prior(1.0)
        self.trajectory_models = dict(models)
        return self

    def _terminal_models_struct(self):
        tm = L.TerminalModels()
        for stem, group, k in self.TRAJECTORY_SLOTS:
            if (group, k) not in self.trajectory_models:
                raise L.EmbError(L.EMB_E_ARG, "trajectory models are not loaded (load_trajectory_models); the public "
                                 "checkout of the reference does not ship them")
            getattr(tm, group)[k] = self.trajectory_models[(group, k)]._h.value
        return tm

    def create_encounters(self, geo, tmax_s: float = 120, seed: int = 0, first_sample: int = 0, device=None,
                          geo_rows: Optional[Sequence[int]] = None, max_attempts: int = 0,
                          out: Optional[TrajectoryResult] = None) -> TrajectoryResult:
        """The batch form of createEncounter.m:1-91 (without the em-core smoothing of :88-89).

        geo: (rows, n) float64, numpy or torch-on-`device`; by default the transposed outInits of `sample`, i.e. one
        row per geometry variable, and `geo_rows` (0-based rows of GEO_FIELDS) is looked up from the labels."""
        lib = L.lib()
        if geo_rows is None:
            geo_rows = []
            for f in self.GEO_FIELDS:
                i = _find(self.labels_initial, '"%s"' % f)
                if not i:
                    raise L.EmbError(L.EMB_E_ARG, "geometry model has no variable %s" % f)
                geo_rows.append(i - 1)
        rows = (C.c_int32 * 12)(*[int(v) for v in geo_rows])
        n = int(geo.shape[1])
        tmax = int(math.floor(tmax_s))
        o = self._opts(max_attempts=max_attempts)
        if device is not None:
            import torch
            dev = torch.device(device)
            o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
            o.stream = torch.cuda.current_stream(dev).cuda_stream
            assert geo.is_cuda and geo.dtype == torch.float64 and geo.is_contiguous()
        else:
            geo = np.ascontiguousarray(geo, dtype=np.float64)
        if out is None:
            out = TrajectoryResult(n=n, tmax=tmax, traj=self._alloc((len(L.TRAJ_FIELDS), 2, 2 * tmax + 1, n), np.float32, device),
                                   len=self._alloc((4, n), np.int16, device))
        lim = (L.DynLimits * 2)()
        L.check(lib.emb_dyn_limits_named(self.acType1.encode(), C.byref(lim[0])))
        L.check(lib.emb_dyn_limits_named(self.acType2.encode(), C.byref(lim[1])))
        tm = self._terminal_models_struct()
        rng = L.Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_sample))
        to = L.TrajOut(_ptr(out.traj), _ptr(out.len))
        L.check(lib.emb_terminal_propagate(C.byref(tm), C.byref(rng), n, _ptr(geo), int(geo.shape[1]), rows, float(tmax_s),
                                           lim, C.byref(o), C.byref(to)))
        return out

    def screen_encounters(self, res: "TrajectoryResult", thresDist_ft: float = 0.0, thresAltLow_ft: float = 0.0, device=None):
        """Batch form of getGeneratedMissDistance (CorTerminalModel.m:117-133), the overlap length of track.m:88 and
        CheckRunwayProximity (CorTerminalModel.m:187-210) on the trajectories of `create_encounters`.
        -> dict(hmd_ft, vmd_ft (n,) float64; tcpa_s, tcpa_index_own, tcpa_index_int, enc_time_s (n,) int16;
                is_close1, is_low1, is_close2, is_low2 (n,) bool)"""
        n = res.n
        o = self._opts()
        if device is not None:
            import torch
            dev = torch.device(device)
            o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
            o.stream = torch.cuda.current_stream(dev).cuda_stream
        hmd, vmd = self._alloc((n,), np.float64, device), self._alloc((n,), np.float64, device)
        tcpa, enc = self._alloc((3, n), np.int16, device), self._alloc((n,), np.int16, device)
        rw = self._alloc((n,), np.uint8, device)
        so = L.ScreenOut(_ptr(hmd), _ptr(vmd), _ptr(tcpa), _ptr(enc), _ptr(rw))
        L.check(L.lib().emb_terminal_screen(_ptr(res.traj), _ptr(res.len), n, float(res.tmax), float(thresDist_ft),
                                            float(thresAltLow_ft), C.byref(o), C.byref(so)))
        return dict(hmd_ft=hmd, vmd_ft=vmd, tcpa_s=tcpa[0], tcpa_index_own=tcpa[1], tcpa_index_int=tcpa[2], enc_time_s=enc,
                    is_close1=(rw & 1) != 0, is_low1=(rw & 2) != 0, is_close2=(rw & 4) != 0, is_low2=(rw & 8) != 0)

    def createEncounter(self, sample_geo: dict, tmax_s: float = 120, seed: int = 0, sample_index: int = 0):
        """createEncounter.m:1 for one `sample_geo` struct (a dict as returned in outSamples) -> traj(1:2)."""
        geo = np.array([[float(sample_geo[f])] for f in self.GEO_FIELDS])
        res = self.create_encounters(geo, tmax_s, seed=seed, first_sample=sample_index, geo_rows=range(12))
        return res.encounter(0)
