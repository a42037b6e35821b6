"""Shared test helpers: model locations, the oracle-side dense view, and the TEST-ONLY host emulation
of the device routines (tests/emu) used by the CPU suite."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from em_model_manned_bayes_b200 import _lib as L  # noqa: E402
from em_model_manned_bayes_b200.model import untile_bins, untile_values  # noqa: E402

# A checkout of the upstream MATLAB project (Airspace-Encounter-Models/em-model-manned-bayes), which this repository does
# not vendor: the sweep over all of its model/*.txt files (more than the packed archive holds) runs only when
# EMB200_REFERENCE_DIR names one.
REF_DIR = os.environ.get("EMB200_REFERENCE_DIR", "")
REF_MODEL_DIR = os.path.join(REF_DIR, "model") if REF_DIR else ""
GOLDEN = os.path.join(ROOT, "tests", "golden")


def have_reference() -> bool:
    return os.path.isdir(REF_MODEL_DIR)


# ---------------------------------------------------------------------------------------------------
def oracle_dense(parms, samples):
    """From oracle UncorSample objects build what emb_sample_tracks returns: bins (n, n_dyn, T) and
    values (n, n_tv, T) plus the variable lists (1-based)."""
    tm = np.asarray(parms.temporal_map)
    dyn = [int(v) for v in tm[:, 0]]
    rates = np.asarray(parms.resample_rates)
    tv = sorted(set(dyn) | {i + 1 for i in range(parms.n_initial) if rates[i] > 0})   # = the gated variables
    bins = np.stack([s.sample_bins[[d - 1 for d in dyn], :] for s in samples]).astype(np.int8)
    vals = np.stack([s.samples[[v - 1 for v in tv], :] for s in samples])
    return bins, vals, dyn, tv


# ---------------------------------------------------------------------------------------------------
_emu = None


def emu_lib():
    """Build (if stale) and load tests/emu/libemb_emu.so."""
    global _emu
    if _emu is not None:
        return _emu
    here = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(here, "libemb_emu.so")
    srcs = [os.path.join(here, "emu.cpp"), os.path.join(ROOT, "em_model_manned_bayes_b200", "csrc", "emb_model.cpp")]
    deps = srcs + [os.path.join(ROOT, "em_model_manned_bayes_b200", "csrc", f) for f in ("emb_device.cuh", "emb_fast.cuh", "emb_initial.cuh", "emb_terminal.cuh", "emb_integrate.cuh", "emb_model.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        cuda_inc = "/usr/local/cuda/include"
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared",
               "-I", cuda_inc] + srcs + ["-o", so]
        subprocess.run(cmd, check=True)
    lib = C.CDLL(so)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    lib.emu_last_error.restype = C.c_char_p
    lib.emu_model_load.argtypes = [C.c_char_p, C.c_int, C.POINTER(i32), i32, C.POINTER(vp)]
    lib.emu_model_free.argtypes = [vp]
    lib.emu_set_prior.argtypes = [vp, C.c_int, C.c_int, C.c_double]
    lib.emu_sample_initial.argtypes = [vp, u64, u64, i64, C.POINTER(L.SampleOpts), vp, vp, vp]
    lib.emu_sample_tracks.argtypes = [vp, u64, u64, i64, i32, C.POINTER(L.SampleOpts), C.POINTER(L.TrackOut)]
    lib.emu_sample_track_events.argtypes = [vp, u64, u64, i64, i32, C.POINTER(L.SampleOpts), i64, vp, vp, C.POINTER(i64)]
    lib.emu_terminal_propagate.argtypes = [C.POINTER(vp), u64, u64, i64, vp, i64, C.POINTER(i32), C.c_double,
                                           C.POINTER(L.DynLimits), i32, vp, vp]
    lib.emu_terminal_screen.argtypes = [vp, vp, i64, C.c_double, C.c_double, C.c_double, vp, vp, vp, vp, vp]
    lib.emu_tracks_integrate.argtypes = [i64, i32, i32, i32, i32, i32, i32, i32] + [C.c_double] * 5 + [vp, vp, vp, vp]
    lib.emu_bearing_cells.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.emu_sincosd.argtypes = [i64, vp, vp, vp]
    lib.emu_sincosd.restype = None
    lib.emu_div_const.argtypes = [i64, vp, vp, vp]
    lib.emu_div_const.restype = None
    lib.emu_use_fast.argtypes = [C.c_int]
    lib.emu_last_fast.restype = C.c_int
    _emu = lib
    return lib


class EmuModel:
    """Host emulation counterpart of em_model_manned_bayes_b200.model.EncounterModel (tests only)."""

    def __init__(self, path, idx_zero=(), overwrite=False):
        self.lib = emu_lib()
        self.h = C.c_void_p()
        idx = (C.c_int32 * max(1, len(idx_zero)))(*idx_zero)
        rc = self.lib.emu_model_load(path.encode(), int(overwrite), idx, len(idx_zero), C.byref(self.h))
        if rc:
            raise L.EmbError(rc, self.lib.emu_last_error().decode())

    def __del__(self):
        try:
            if self.h.value:
                self.lib.emu_model_free(self.h)
                self.h = C.c_void_p()
        except Exception:
            pass

    def set_prior(self, which, kind, value):
        rc = self.lib.emu_set_prior(self.h, which, kind, value)
        if rc:
            raise L.EmbError(rc, self.lib.emu_last_error().decode())

    @staticmethod
    def opts(n_initial, start=None, **kw):
        o = L.SampleOpts()
        for i in range(L.EMB_MAX_VARS):
            o.box_lo[i], o.box_hi[i] = -np.inf, np.inf
        o.device = -1
        if start is not None:
            for i, s in enumerate(start):
                o.start[i] = 0 if s is None else int(s)
        for k, v in kw.items():
            if k == "layers":
                v = np.asarray(v, dtype=np.float64).reshape(-1, 2)
                o.n_layers = v.shape[0]
                for r in range(v.shape[0]):
                    o.layers[r][0], o.layers[r][1] = v[r, 0], v[r, 1]
            elif k in ("box_lo", "box_hi"):
                for i, x in enumerate(v):
                    getattr(o, k)[i] = float(x)
            else:
                setattr(o, k, v)
        return o

    def sample_initial(self, n_initial, n, seed, first, opts):
        bins = np.zeros((n_initial, n), dtype=np.int8)
        vals = np.zeros((n_initial, n), dtype=np.float64)
        att = np.zeros(n, dtype=np.uint16)
        rc = self.lib.emu_sample_initial(self.h, seed, first, n, C.byref(opts), bins.ctypes.data, vals.ctypes.data,
                                         att.ctypes.data)
        if rc:
            raise L.EmbError(rc, self.lib.emu_last_error().decode())
        return bins.T, vals.T, att

    def sample_events(self, n, T, seed, first, opts, capacity=None):
        """-> (events structured array, offsets int64 [n+1])"""
        cap = capacity if capacity is not None else n * (8 * T + 8)
        ev = np.zeros(max(cap, 1), dtype=L.EVENT_DTYPE)
        off = np.zeros(n + 1, dtype=np.int64)
        total = C.c_int64(0)
        rc = self.lib.emu_sample_track_events(self.h, seed, first, n, T, C.byref(opts), cap, ev.ctypes.data, off.ctypes.data,
                                              C.byref(total))
        if rc:
            raise L.EmbError(rc, self.lib.emu_last_error().decode())
        return ev[:total.value], off

    def sample_tracks(self, n_initial, n_dyn, n_tv, n, T, seed, first, opts, hist=False):
        nch, npad = (T + 3) // 4, (n + 127) // 128 * 128
        bins = np.zeros(n_dyn * nch * npad * 4, dtype=np.int8)
        vals = np.zeros(n_tv * nch * npad * 4, dtype=np.float32)
        ib = np.zeros((n_initial, n), dtype=np.int8)
        iv = np.zeros((n_initial, n), dtype=np.float64)
        att = np.zeros(n, dtype=np.uint16)
        hi = np.zeros((n_initial, 64), dtype=np.uint64) if hist else None
        ht = np.zeros((n_dyn, 64), dtype=np.uint64) if hist else None
        to = L.TrackOut(bins.ctypes.data, vals.ctypes.data, ib.ctypes.data, iv.ctypes.data, att.ctypes.data,
                        hi.ctypes.data if hist else None, ht.ctypes.data if hist else None)
        rc = self.lib.emu_sample_tracks(self.h, seed, first, n, T, C.byref(opts), C.byref(to))
        if rc:
            raise L.EmbError(rc, self.lib.emu_last_error().decode())
        return dict(bins=untile_bins(bins, n_dyn, n, T), values=untile_values(vals, n_tv, n, T), init_bins=ib.T,
                    init_values=iv.T, attempts=att, hist_initial=hi, hist_transition=ht)
