"""sample2track.m:1-300 -- first-order tracks from sampled initial conditions and per-second rates, on top of the C ABI.

  integrate_tracks(model, res)                  the per-track loop of sample2track.m:188-244 on a TrackResult that is
                                                still in HBM (or in host memory): (xyz (3, T+1, n) float32, is_good (n,))
  parse_table(text, cols, device=None)          the body of a decimal text table (initial.txt, transition.txt) parsed on
                                                the device, bit for bit what np.loadtxt / float() give (emb_parse_table)
  format_tracks_csv(xyz, mask, device=None)     the CSV rows "%d,%.0f,%.0f,%.0f" of every unmasked track, formatted on the
                                                device byte for byte as Python's '%' (emb_format_tracks_csv)
  sample2track(parameters_filename, initial_filename, transition_filename, ...)
                                                the reference's file-to-file driver: reads the two text files em_sample
                                                wrote, parses, groups, integrates and formats on the GPU, writes
                                                BAYES_t*_id*_alt*_speed*.csv into the same G*/A*/<alt>ft directory tree
                                                (:143-178, :246-290); the host only reads and writes the files

Differences from the reference, all outside the integration itself: `randperm` (when the initial file holds more than
num_max_tracks tracks, :77-79) uses numpy's generator seeded with rng_seed, and plotting (:220-232) is not offered."""
from __future__ import annotations

import ctypes as C
import math
import os
import re
from typing import Optional

import numpy as np

from . import _lib as L
from .model import EncounterModel, TrackResult, _ptr, tile

FT_PER_NM = 1852.0 / 0.3048           # unitsratio('ft', 'nm')


def make_valid_name(label: str) -> str:
    """matlab.lang.makeValidName(erase(label, {'"', '\\'})) for the labels of the shipped models
    ('"\\dot v"' -> 'dotV', '"\\dot h(t+1)"' -> 'dotH_t_1_')."""
    s = label.replace('"', "").replace("\\", "")
    s = re.sub(r"\s+([a-zA-Z])", lambda m: m.group(1).upper(), s.strip())   # whitespace removed, next letter upper-cased
    s = re.sub(r"\s+", "", s)
    s = re.sub(r"[^A-Za-z0-9_]", "_", s)
    if not re.match(r"[A-Za-z]", s):
        s = "x" + s
    return s


def _find(names, name):
    return names.index(name) + 1 if name in names else 0


def integrate_opts(model: EncounterModel, label_initial_altitude="L", label_initial_speed="v",
                   label_initial_acceleration="dotV", label_initial_vertrate="dotH", label_initial_turnrate="dotPsi"):
    """sample2track.m:81-141: column lookup, unit ratios and speed bounds."""
    names = [make_valid_name(l) for l in model.labels_initial]
    o = L.IntegrateOpts()
    o.idx_altitude, o.idx_speed = _find(names, label_initial_altitude), _find(names, label_initial_speed)
    o.idx_acceleration = _find(names, label_initial_acceleration)
    o.idx_vertrate, o.idx_turnrate = _find(names, label_initial_vertrate), _find(names, label_initial_turnrate)
    if not all((o.idx_altitude, o.idx_speed, o.idx_acceleration, o.idx_vertrate, o.idx_turnrate)):
        raise L.EmbError(L.EMB_E_ARG, "sample2track: the model lacks one of the variables L, v, dotV, dotH, dotPsi")
    o.ur_speed, o.ur_vertrate, o.ur_heading = FT_PER_NM / 3600.0, 1.0 / 60.0, 1.0             # :108-125
    b = model.boundaries[o.idx_speed - 1]
    o.min_speed, o.max_speed = float(b[0]) * o.ur_speed, float(b[-1]) * o.ur_speed           # :98-99, :140-141
    o.mem, o.device, o.stream = L.EMB_MEM_HOST, -1, None
    return o


def integrate_tracks(model: EncounterModel, res: TrackResult, opts: Optional[L.IntegrateOpts] = None, device=None,
                     want_xyz: bool = True):
    """sample2track.m:188-244 for every track of `res` (dense compact output of sample_tracks).
    Returns (xyz (3, T+1, n) float32: x_ft, y_ft, z_ft at time_s = 0..T, is_good (n,) uint8)."""
    o = opts if opts is not None else integrate_opts(model)
    n, T = res.n, res.T
    if device is not None:
        import torch
        dev = torch.device(device)
        o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
        o.stream = torch.cuda.current_stream(dev).cuda_stream
        xyz = torch.empty((3, T + 1, n), dtype=torch.float32, device=dev) if want_xyz else None
        good = torch.empty((n,), dtype=torch.uint8, device=dev)
    else:
        xyz = np.empty((3, T + 1, n), dtype=np.float32) if want_xyz else None
        good = np.empty((n,), dtype=np.uint8)
    L.check(L.lib().emb_tracks_integrate(model._h, n, T, _ptr(res.init_values), _ptr(res.values_tiled), C.byref(o),
                                         _ptr(xyz), _ptr(good)))
    return xyz, good


def sample_tracks_xyz(model: EncounterModel, n: int, T: int, seed: int = 0, first_sample: int = 0, sample_opts=None,
                      opts: Optional[L.IntegrateOpts] = None, device=None, want_xyz: bool = True, dense: Optional[TrackResult] = None):
    """Sampling and the Euler loop of sample2track.m:188-244 in ONE kernel pass (emb200.h: emb_sample_tracks_xyz): the same
    (xyz, is_good) as `integrate_tracks(model, model.sample_tracks(...))` without the dense tiles' round trip through HBM.
    `sample_opts`: e.g. `UncorEncounterModel.uncor_opts()`; `dense`: a TrackResult whose buffers are filled as well."""
    io = opts if opts is not None else integrate_opts(model)
    so = sample_opts if sample_opts is not None else model._opts()
    if device is not None:
        import torch
        dev = torch.device(device)
        so.mem, so.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
        so.stream = torch.cuda.current_stream(dev).cuda_stream
        xyz = torch.empty((3, T + 1, n), dtype=torch.float32, device=dev) if want_xyz else None
        good = torch.empty((n,), dtype=torch.uint8, device=dev)
    else:
        xyz = np.empty((3, T + 1, n), dtype=np.float32) if want_xyz else None
        good = np.empty((n,), dtype=np.uint8)
    to = None
    if dense is not None:
        to = L.TrackOut(_ptr(dense.bins_tiled), _ptr(dense.values_tiled), _ptr(dense.init_bins), _ptr(dense.init_values),
                        _ptr(dense.attempts), None, None)
    rng = L.Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_sample))
    L.check(L.lib().emb_sample_tracks_xyz(model._h, C.byref(rng), n, T, C.byref(so), C.byref(io),
                                          C.byref(to) if to is not None else None, _ptr(xyz), _ptr(good)))
    return xyz, good


def _torch_call(arrays, device):
    """Options and buffer kind of a text call: torch CUDA tensors in -> device buffers on their device (None: the host);
    numpy or bytes in -> host buffers, computed on `device` (CUDA ordinal or torch device; default the current one)."""
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem, o.device, o.stream = L.EMB_MEM_HOST, -1, None
    a = arrays[0]
    if not isinstance(a, (np.ndarray, bytes, bytearray, memoryview)):
        import torch
        dev = a.device
        if dev.type != "cuda" or any(x.device != dev for x in arrays):
            raise L.EmbError(L.EMB_E_ARG, "tensors must all be on one CUDA device (or pass numpy arrays)")
        o.mem, o.device = L.EMB_MEM_DEVICE, dev.index if dev.index is not None else torch.cuda.current_device()
        o.stream = torch.cuda.current_stream(dev).cuda_stream
        return o, dev
    if device is not None:
        import torch
        dev = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        o.device = dev.index if dev.index is not None else -1
    return o, None


def parse_table(text, cols: int, device=None):
    """The body of a decimal text table (no header line) -> (rows, cols) float64, parsed on the device (emb200.h:
    emb_parse_table): the lines and fields of np.loadtxt, blank lines skipped, every value bit for bit Python's float() of its
    field.  `text`: bytes / numpy uint8 (numpy out, computed on `device`) or a uint8 torch CUDA tensor (a tensor on its device
    out).  A malformed field, a wrong field count or a value beyond DBL_MAX raises EmbError(EMB_E_ARG) naming the line."""
    o, like = _torch_call([text], device)
    if like is None:
        t = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else np.ascontiguousarray(text, dtype=np.uint8)
        nbytes = int(t.shape[0])
    else:
        import torch
        t = text.contiguous().view(torch.uint8).reshape(-1)
        nbytes = int(t.numel())
    ptr = (t.ctypes.data if nbytes else None) if like is None else (t.data_ptr() if nbytes else None)
    lib = L.lib()
    rows, bad = C.c_int64(0), C.c_int64(0)
    rc = lib.emb_parse_table(ptr, nbytes, int(cols), C.byref(o), 0, None, C.byref(rows), C.byref(bad))   # sizes the call
    if rc == L.EMB_E_LIMIT:
        n = int(rows.value)
        if like is None:
            out = np.empty((n, int(cols)), dtype=np.float64)
        else:
            import torch
            out = torch.empty((n, int(cols)), dtype=torch.float64, device=like)
        rc = lib.emb_parse_table(ptr, nbytes, int(cols), C.byref(o), n, _ptr(out), C.byref(rows), C.byref(bad))
        L.check(rc)
        return out
    L.check(rc)
    if like is None:
        return np.empty((0, int(cols)), dtype=np.float64)
    import torch
    return torch.empty((0, int(cols)), dtype=torch.float64, device=like)


CSV_ROW_GUESS = 40   # bytes per CSV row to try first: within 10^6 ft and T < 10^4 a row has at most 32 (else the call is retried)


def format_tracks_csv(xyz, mask=None, device=None):
    """The CSV rows of sample2track.m:246-290 without the header line, formatted on the device (emb200.h:
    emb_format_tracks_csv): for each track k with mask[k] != 0 (every track if mask is None), T+1 rows
    "%d,%.0f,%.0f,%.0f\\n" % (t, x, y, z), t = 0 .. T, byte for byte as Python's '%' prints them.  `xyz`: (3, T+1, n) float32,
    the layout of `integrate_tracks`; `mask`: (n,) uint8 or bool.  Returns (text uint8, offsets int64 [n+1]): track k is
    text[offsets[k]:offsets[k+1]], empty when masked.  numpy in, numpy out (computed on `device`); torch CUDA tensors in, tensors
    on their device out."""
    o, like = _torch_call([xyz] + ([mask] if mask is not None else []), device)
    if xyz.shape[0] != 3 or len(xyz.shape) != 3:
        raise L.EmbError(L.EMB_E_ARG, "format_tracks_csv: xyz must be (3, T+1, n)")
    T, n = int(xyz.shape[1]) - 1, int(xyz.shape[2])
    if like is None:
        x = np.ascontiguousarray(xyz, dtype=np.float32)
        mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        off = np.zeros(n + 1, dtype=np.int64)
        empty = lambda k: np.empty((k,), dtype=np.uint8)
    else:
        import torch
        x = xyz.to(torch.float32).contiguous()
        mk = None if mask is None else mask.to(torch.uint8).contiguous()
        off = torch.zeros(n + 1, dtype=torch.int64, device=like)
        empty = lambda k: torch.empty((k,), dtype=torch.uint8, device=like)
    if mk is not None and int(mk.shape[0]) != n:
        raise L.EmbError(L.EMB_E_ARG, "format_tracks_csv: mask must have n entries")
    lib = L.lib()
    total = C.c_int64(0)
    cap = n * (T + 1) * CSV_ROW_GUESS
    text = empty(cap)
    rc = lib.emb_format_tracks_csv(n, T, _ptr(x), _ptr(mk), C.byref(o), cap, _ptr(text), _ptr(off), C.byref(total))
    if rc == L.EMB_E_LIMIT and int(total.value) > cap:
        cap = int(total.value)
        text = empty(cap)
        rc = lib.emb_format_tracks_csv(n, T, _ptr(x), _ptr(mk), C.byref(o), cap, _ptr(text), _ptr(off), C.byref(total))
    L.check(rc)
    return text[:int(total.value)], off


def _read_body(path):
    """The bytes of a text file after its header line, which ends where a universal-newline readline() ends it (CRLF, CR
    or LF): what np.loadtxt read after `f.readline()` in the host driver this replaces."""
    data = bytearray(os.path.getsize(path))
    with open(path, "rb") as f:
        f.readinto(data)
    m = re.search(rb"\r\n|\r|\n", data)
    return data, (m.end() if m else len(data))


def _to_device(path, dev):
    import torch
    data, start = _read_body(path)
    if start == len(data):
        return torch.empty((0,), dtype=torch.uint8, device=dev)
    return torch.frombuffer(data, dtype=torch.uint8, offset=start).to(dev)


def sample2track(parameters_filename: str, initial_filename: str, transition_filename: str, num_max_tracks: int = 10000,
                 out_dir_parent: str = "output/tracks", isOverwriteZeroBoundaries: bool = False, idxZeroBoundaries=(1, 2, 3),
                 rng_seed: int = 42, label_initial_geographic="G", label_initial_airspace="A", device=None, **labels):
    """-> (is_good (num_tracks,) bool, T_initial (num_tracks, 1 + n_initial) with the unit conversions of :128-131).
    The two files are parsed, grouped by id, integrated and formatted on `device` (default: the current CUDA device); the host
    reads the files, computes the directory and file names from one value per track, and writes the CSV files."""
    import torch
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    model = EncounterModel(parameters_filename, idxZeroBoundaries=idxZeroBoundaries,
                           isOverwriteZeroBoundaries=isOverwriteZeroBoundaries)
    o = integrate_opts(model, **labels)
    names_init = [make_valid_name(l) for l in model.labels_initial]
    dyn_t = [int(v) for v in model.temporal_map[:, 0]]
    Ti = parse_table(_to_device(initial_filename, dev), 1 + model.n_initial)             # id, initial variables
    Tt = parse_table(_to_device(transition_filename, dev), 2 + len(dyn_t))              # id, t, dynamic variables (temporal_map order)
    if Ti.shape[0] > num_max_tracks:                                      # :77-79
        keep = np.sort(np.random.default_rng(rng_seed).permutation(Ti.shape[0])[:num_max_tracks])
        Ti = Ti[torch.from_numpy(keep).to(dev)]
    n = int(Ti.shape[0])
    ids = Ti[:, 0].to(torch.int64).to(torch.float64)                      # truncated like astype(np.int64), compared as doubles
    key, order = torch.sort(Tt[:, 0], stable=True)
    Tt = Tt[order]
    first = torch.searchsorted(key, ids, side="left")
    last = torch.searchsorted(key, ids, side="right")
    cnt = (last - first).cpu().numpy()
    T = int(cnt[0])
    if T < 1 or np.any(cnt != T):
        raise L.EmbError(L.EMB_E_ARG, "sample2track: every track needs the same number of transition rows")
    rows = (first[:, None] + torch.arange(T, device=dev)[None, :]).reshape(-1)
    upd = Tt[rows, 2:].reshape(n, T, len(dyn_t))                          # (n, T, n_dyn) float64
    tv = list(model.timevarying_vars)
    dense = torch.zeros((n, len(tv), T), dtype=torch.float32, device=dev)
    for k, v in enumerate(dyn_t):
        dense[:, tv.index(v), :] = upd[:, :, k]                           # decimal -> double -> float, as np.float32 assigns
    res = TrackResult(n=n, T=T, dyn_vars=dyn_t, tv_vars=tv, bins_tiled=None, values_tiled=tile(dense), init_bins=None,
                      init_values=Ti[:, 1:].T.contiguous(), attempts=None)
    xyz, good = integrate_tracks(model, res, opts=o, device=dev)
    text, offsets = format_tracks_csv(xyz, good)
    Ti = Ti.cpu().numpy()
    is_good = good.cpu().numpy().astype(bool)
    z0s = xyz[2, 0].cpu().numpy()
    text, offsets = text.cpu().numpy(), offsets.cpu().numpy()
    # ---- output tree and files (:143-178, :246-290)
    b_alt = model.boundaries[o.idx_altitude - 1]
    min_alt, max_alt = float(b_alt[0]), float(b_alt[-1])
    Ls = np.arange(math.floor(min_alt - 50) if min_alt % 100 else min_alt, max_alt + 200 + 1e-9, 100.0)      # :151-158
    if Ls[0] < 0:
        Ls[0] = 0
    iG, iA = _find(names_init, label_initial_geographic), _find(names_init, label_initial_airspace)
    speed0 = Ti[:, o.idx_speed] * o.ur_speed
    view = memoryview(text)
    for k in np.nonzero(is_good)[0]:
        z0 = float(z0s[k])
        parts = []
        if iG:
            parts.append("G%d" % int(Ti[k, iG]))
        if iA:
            parts.append("A%d" % int(Ti[k, iA]))
        j = int(np.searchsorted(Ls, z0, side="right")) - 1                # discretize(z_ft(1), L) (:266)
        parts.append("%dft" % int(Ls[min(max(j, 0), len(Ls) - 2)]))
        d = os.path.join(out_dir_parent, *parts)
        os.makedirs(d, exist_ok=True)
        name = "BAYES_t%d_id%d_alt%d_speed%d.csv" % (T, k + 1, int(math.floor(z0 + 0.5)), int(math.floor(speed0[k] + 0.5)))
        with open(os.path.join(d, name), "wb") as f:
            f.write(b"time_s,x_ft,y_ft,z_ft\n")
            f.write(view[offsets[k]:offsets[k + 1]])
    Tc = Ti.copy()
    Tc[:, o.idx_speed] *= o.ur_speed
    Tc[:, o.idx_acceleration] *= o.ur_speed
    Tc[:, o.idx_vertrate] *= o.ur_vertrate
    return is_good, Tc
