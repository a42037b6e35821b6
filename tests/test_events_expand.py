"""CPU suite for out_samples and the control rows computed from event lists (emb_track_events_expand[_packed]): the per-track
routines of emb_events_expand.cuh, run on the host by the TEST-ONLY emulation in tests/emu/emu_events_expand.cpp, against the
oracle's events2samples / events2controls (oracle/sampler.py), model.py's expand_events / controls_of, the out_EME transform
of UncorEncounterModel.sample and PackedEventResult.decode; the refusals of the C ABI that need no device."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import cases
from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import (EncounterModel, PackedEventResult, UncorEncounterModel, controls_of,
                                              expand_events)
from helpers import ROOT
from oracle import sampler as OS

# status bits of emb_loglik.cuh / emb_loglik_events.cuh that the expansion raises
BAD_BIN, BAD_VAR, BAD_OFFSETS = 1, 4, 16

_ee = None


def _lib():
    """Build (once per process, into a temporary directory: the tree may be read-only) and load the emulation."""
    global _ee
    if _ee is not None:
        return _ee
    out = os.path.join(tempfile.mkdtemp(prefix="emb_events_expand_emu_"), "libemb_events_expand_emu.so")
    srcs = [os.path.join(ROOT, "tests", "emu", "emu_loglik.cpp"), os.path.join(ROOT, "tests", "emu", "emu_events_expand.cpp"),
            os.path.join(ROOT, "em_model_manned_bayes_b200", "csrc", "emb_model.cpp")]
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared",
                    "-I", "/usr/local/cuda/include"] + srcs + ["-o", out], check=True)
    lib = C.CDLL(out)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.ll_last_error.restype = C.c_char_p
    lib.ll_model_load.argtypes = [C.c_char_p, C.c_int, C.POINTER(i32), i32, C.POINTER(vp)]
    lib.ll_model_free.argtypes = [vp]
    lib.ee_expand.argtypes = [vp, i64, i32, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    _ee = lib
    return lib


class EmuModel:
    """A model loaded into the emulation (tests only), beside the library's view of the same file and zero-bin options."""

    def __init__(self, path, idx_zero=(), overwrite=False, uncor=False):
        self.lib = _lib()
        self.h = C.c_void_p()
        idx = (C.c_int32 * max(1, len(idx_zero)))(*idx_zero)
        rc = self.lib.ll_model_load(path.encode(), int(overwrite), idx, len(idx_zero), C.byref(self.h))
        assert rc == 0, self.lib.ll_last_error()
        if uncor:
            self.m = UncorEncounterModel(path, idxZeroBoundaries=idx_zero, isOverwriteZeroBoundaries=overwrite)
        else:
            self.m = EncounterModel(path, idxZeroBoundaries=idx_zero, isOverwriteZeroBoundaries=overwrite)

    def __del__(self):
        try:
            if self.h.value:
                self.lib.ll_model_free(self.h)
                self.h = C.c_void_p()
        except Exception:
            pass


def rows_8byte(dt, var, bins, value):
    ev = np.zeros(len(dt), dtype=L.EVENT_DTYPE)
    ev["dt"], ev["var"], ev["bin"], ev["value"] = dt, var, bins, value
    return ev


def rows_packed(em, dt, var, bins, frac):
    """the 5-byte rows of emb_sample_track_events_packed for the same (dt, var, bin) rows and 23-bit fractions"""
    gord_of = {int(v): k + 1 for k, v in enumerate(em.m.gated_vars)}
    dt, var, bins, frac = (np.asarray(a, dtype=np.int64) for a in (dt, var, bins, frac))
    gord = np.array([gord_of[int(v)] if v > 0 else 0 for v in var], dtype=np.int64)
    words = np.where(gord > 0, frac | ((bins - 1) << 23), 0) | (gord << 27) | ((dt >> 8) << 30)
    return words.astype(np.uint32), (dt & 255).astype(np.uint8)


def decode(em, words, dts, T):
    """values of packed rows as PackedEventResult.decode gives them"""
    r = PackedEventResult(n=0, T=T, words=words, dts=dts, offsets=None, init_bins=None, init_values=None, attempts=None,
                          total=len(words), gated_vars=list(em.m.gated_vars), boundaries=em.m.boundaries,
                          zero_bins=em.m.zero_bins)
    return r.decode()[3]


def resolve(em, spec):
    """spec None (events2controls.m: temporal_map(:,1), unscaled) or (vars 1-based, mul, div) -> 0-based vars, mul, div"""
    if spec is None:
        v = [int(x) - 1 for x in np.asarray(em.m.temporal_map)[:, 0]]
        return v, [1.0] * len(v), [1.0] * len(v)
    return [int(x) - 1 for x in spec[0]], list(spec[1]), list(spec[2])


def emu_expand(em, init_values, rows, dts, offsets, T, packed, spec=None, status=0, samples=True):
    """init_values (n, n_initial) -> (samples (n, T, n_initial) or None, [control matrix per track]); asserts the status"""
    iv = np.ascontiguousarray(np.asarray(init_values, dtype=np.float64).T)
    n, ni = iv.shape[1], iv.shape[0]
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    rows = rows if len(rows) else np.zeros(1, dtype=rows.dtype)
    dts = dts if dts is not None and len(dts) else np.zeros(1, dtype=np.uint8)
    vars_, mul, div = resolve(em, spec)
    k = len(vars_)
    ctl_off = np.zeros(n + 1, dtype=np.int64)
    # the count pass alone first (controls NULL), then both passes into buffers of the counted size
    cv, cm, cd = (np.array(vars_, dtype=np.int32), np.array(mul), np.array(div))
    lib = _lib()
    args = (em.h, n, T, iv.ctypes.data, rows.ctypes.data, dts.ctypes.data, off.ctypes.data, int(packed), k, cv.ctypes.data,
            cm.ctypes.data, cd.ctypes.data)
    got = lib.ee_expand(*args, None, None, ctl_off.ctypes.data)
    if got:
        assert got == status, "status %d, expected %d" % (got, status)
        return None, None
    total = int(ctl_off[n])
    ctl = np.full((max(total, 1), 1 + k), np.nan)
    smp = np.full((n, T, ni), np.nan) if samples else None
    got = lib.ee_expand(*args, None if smp is None else smp.ctypes.data, ctl.ctypes.data, ctl_off.ctypes.data)
    assert got == status, "status %d, expected %d" % (got, status)
    return smp, [ctl[ctl_off[s]:ctl_off[s + 1]] for s in range(n)]


def oracle_tracks(init_values, dt, var, value, offsets):
    """(init row, [[dt, var, value], ...]) per track, for the oracle's per-track statements"""
    ev = np.stack([np.asarray(dt, np.float64), np.asarray(var, np.float64), np.asarray(value, np.float64)], axis=1)
    return [(np.asarray(init_values[s], np.float64), [list(r) for r in ev[offsets[s]:offsets[s + 1]]])
            for s in range(len(offsets) - 1)]


def assert_bits(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, "%s: shape %s, expected %s" % (what, got.shape, want.shape)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), "%s differ" % what


def check_against_host(em, init_values, dt, var, value, off, T, smp, ctl, full_lists=True):
    """emulated samples and plain controls against expand_events / controls_of and the oracle's per-track statements"""
    n = len(off) - 1
    if len(dt):
        dense = expand_events(init_values, dt, var, value, off, T)                 # (n, n_initial, T)
    else:
        dense = np.repeat(np.asarray(init_values, np.float64)[:, :, None], T, axis=2)
    assert_bits(smp, dense.transpose(0, 2, 1), "samples vs expand_events")
    tm = np.asarray(em.m.temporal_map)
    if full_lists:   # sum(dt) == T in every list
        want = controls_of(dense, dt, off, tm[:, 0] - 1)
        for s in range(n):
            assert_bits(ctl[s], want[s], "controls vs controls_of (track %d)" % s)
    for s, (init, ev) in enumerate(oracle_tracks(init_values, dt, var, value, off)):
        if full_lists:
            assert_bits(smp[s].T, OS.events2samples(init, ev), "samples vs oracle events2samples (track %d)" % s)
        assert_bits(ctl[s], OS.events2controls(init, ev, tm), "controls vs oracle events2controls (track %d)" % s)


def golden_model(model_paths, name):
    c = cases.TRACK_CASES[name]
    ow = tuple(c.get("overwrite", ()))
    idx = ow or ((1, 2, 3) if c["uncor"] else ())
    return c, EmuModel(model_paths[c["model"]], idx_zero=idx, overwrite=bool(ow), uncor=c["uncor"])


def eme_want(em, init_values, dt, var, value, off, T):
    """the out_EME event matrices exactly as UncorEncounterModel.sample builds them"""
    m = em.m
    dense = expand_events(init_values, dt, var, value, off, T)
    ctl = controls_of(dense, dt, off, [v - 1 for v in (m.idxDH, m.idxDPsi, m.idxDV)])
    for c in ctl:
        c[:, 1] /= 60.0
        c[:, 2] *= math.pi / 180.0
        c[:, 3] *= 1.68780972222222
    return ctl


@pytest.mark.parametrize("name", sorted(cases.TRACK_CASES))
def test_golden_lists_8byte_rows(model_paths, golden, name):
    c, em = golden_model(model_paths, name)
    g, T = golden[name], c["T"]
    ev, off = g["events"], g["event_offsets"]
    dt, var = ev[:, 0].astype(np.int64), ev[:, 1].astype(np.int64)
    value = ev[:, 2].astype(np.float32).astype(np.float64)           # what an 8-byte row carries
    rows = rows_8byte(dt, var, g["event_bins"].astype(np.int64), value)
    smp, ctl = emu_expand(em, g["init_values"], rows, None, off, T, packed=False)
    check_against_host(em, g["init_values"], dt, var, value, off, T, smp, ctl)
    if isinstance(em.m, UncorEncounterModel) and em.m.idxDH and em.m.idxDPsi and em.m.idxDV:
        _, eme = emu_expand(em, g["init_values"], rows, None, off, T, packed=False, spec=em.m.out_eme_spec(), samples=False)
        want = eme_want(em, g["init_values"], dt, var, value, off, T)
        for s in range(len(off) - 1):
            assert_bits(eme[s], want[s], "out_EME rows (track %d)" % s)


@pytest.mark.parametrize("name", sorted(cases.TRACK_CASES))
def test_golden_lists_packed_rows(model_paths, golden, name):
    c, em = golden_model(model_paths, name)
    g, T = golden[name], c["T"]
    if len(em.m.gated_vars) > 7 or T > 1023:
        pytest.skip("outside the packed format")
    ev, off = g["events"], g["event_offsets"]
    dt, var, bins = ev[:, 0].astype(np.int64), ev[:, 1].astype(np.int64), g["event_bins"].astype(np.int64)
    frac = np.random.default_rng(len(name)).integers(0, 1 << 23, len(dt))
    words, dts = rows_packed(em, dt, var, bins, frac)
    value = decode(em, words, dts, T)
    smp, ctl = emu_expand(em, g["init_values"], words, dts, off, T, packed=True)
    check_against_host(em, g["init_values"], dt, var, value, off, T, smp, ctl)
    if isinstance(em.m, UncorEncounterModel) and em.m.idxDH and em.m.idxDPsi and em.m.idxDV:
        _, eme = emu_expand(em, g["init_values"], words, dts, off, T, packed=True, spec=em.m.out_eme_spec(), samples=False)
        want = eme_want(em, g["init_values"], dt, var, value, off, T)
        for s in range(len(off) - 1):
            assert_bits(eme[s], want[s], "out_EME rows (track %d)" % s)


def test_packed_values_equal_decode(model_paths):
    """every bin of every gated variable of the flagship model, each visible in its own column: the samples hold dedisc()
    of the packed rows, which must be PackedEventResult.decode bit for bit (zero bins and '*' variables included)"""
    em = EmuModel(model_paths["uncor_allcode_fwsingle_v1"], idx_zero=(1, 2, 3), uncor=True)
    rng = np.random.default_rng(5)
    rows = [(1, v, b) for v in em.m.gated_vars for b in range(1, int(em.m.r_initial[v - 1]) + 1) for _ in range(3)]
    rows.append((1, 0, 0))
    dt, var, bins = (np.array(c, dtype=np.int64) for c in zip(*rows))
    frac = rng.integers(0, 1 << 23, len(dt))
    frac[::3] = 0
    frac[1::3] = (1 << 23) - 1
    words, dts = rows_packed(em, dt, var, bins, frac)
    T = len(rows)
    init = np.zeros((1, em.m.n_initial))
    smp, _ = emu_expand(em, init, words, dts, np.array([0, len(rows)]), T, packed=True)
    value = decode(em, words, dts, T)
    got = smp[0, np.arange(len(rows) - 1) + 1, var[:-1] - 1]
    assert_bits(got, value[:-1], "dedisc() vs PackedEventResult.decode")


# ---- edge lists on a hand-made model ------------------------------------------------------------------------------------
# initial A (r=2, '*') -> B (r=3, edges -10 0 10 20, zero bin 2); transition B(t) -> B(t+1); both resampled, so both gated.
EDGE_MODEL = """# labels_initial
"A", "B"
# G_initial
0 1
0 0
# r_initial
2 3
# N_initial
3 1 1 0 4 0 0 0
# labels_transition
"A", "B(t)", "B(t+1)"
# G_transition
0 0 0
0 0 1
0 0 0
# r_transition
2 3 3
# N_transition
5 5 0 1 2 3 0 0 0
# boundaries
*
-10 0 10 20
# resample_rates
0.1 0.1
"""


@pytest.fixture
def edge(tmp_path):
    f = tmp_path / "edge.txt"
    f.write_text(EDGE_MODEL)
    return str(f), EmuModel(str(f), idx_zero=(2,))


def lists(tracks):
    """[[(dt, var, bin), ...] per track] -> dt, var, bin, offsets"""
    rows = [r for t in tracks for r in t]
    off = np.concatenate(([0], np.cumsum([len(t) for t in tracks]))).astype(np.int64)
    a = np.array(rows, dtype=np.int64).reshape(-1, 3)
    return a[:, 0], a[:, 1], a[:, 2], off


EDGE_LISTS = {
    # (init values (A, B), rows (dt, var, bin), T)
    "several rows of one variable in one second": ((1, 3.5), [(2, 2, 2), (0, 2, 3), (0, 2, 1), (0, 2, 3), (3, 0, 0)], 5),
    "rows at column >= T": ((1, -4.0), [(1, 2, 3), (3, 2, 1), (1, 2, 3), (0, 1, 2), (2, 0, 0)], 4),
    "sum dt < T": ((2, 7.0), [(1, 2, 1), (1, 2, 3)], 7),
    "closing row with dt = 0": ((1, 1.0), [(2, 2, 3), (3, 1, 2), (0, 0, 0)], 5),
    "closing row only": ((2, -1.5), [(6, 0, 0)], 6),
    "dt = 0 rows at column 0": ((1, 2.0), [(0, 2, 3), (0, 1, 2), (0, 2, 1), (2, 2, 2), (2, 0, 0)], 4),
    "T = 1": ((1, 2.0), [(1, 2, 1), (1, 0, 0)], 1),
    "change back within a second": ((1, 5.0), [(2, 2, 3), (0, 2, 1), (3, 0, 0)], 5),
    "more than a warp of rows": ((1, 0.25), [(k % 3, 1 + k % 2, 1 + (k // 2) % 2) for k in range(75)] + [(2, 0, 0)], 60),
}


@pytest.mark.parametrize("packed", [False, True], ids=["rows8", "packed"])
@pytest.mark.parametrize("case", sorted(EDGE_LISTS))
def test_edge_lists(edge, case, packed):
    _, em = edge
    init, rows, T = EDGE_LISTS[case]
    iv = np.array([init], dtype=np.float64)
    dt, var, bins, off = lists([rows])
    frac = (np.arange(len(dt)) * 1234567) & 0x7FFFFF
    words, dts = rows_packed(em, dt, var, bins, frac)
    value = decode(em, words, dts, T)
    rows8 = rows_8byte(dt, var, bins, value.astype(np.float32))
    if packed:
        smp, ctl = emu_expand(em, iv, words, dts, off, T, packed=True)
    else:
        value = value.astype(np.float32).astype(np.float64)
        smp, ctl = emu_expand(em, iv, rows8, None, off, T, packed=False)
    check_against_host(em, iv, dt, var, value, off, T, smp, ctl, full_lists=int(dt.sum()) == T)


def test_empty_tracks_and_ragged_batch(edge):
    _, em = edge
    tracks = [[], [(2, 2, 3), (3, 0, 0)], [], [(1, 1, 2), (0, 2, 1), (9, 0, 0)], []]
    iv = np.array([[1, 4.0], [2, -3.0], [1, 0.5], [2, 8.0], [1, 1.0]])
    dt, var, bins, off = lists(tracks)
    for T in (1, 5, 12):
        words, dts = rows_packed(em, dt, var, bins, np.full(len(dt), 77))
        value = decode(em, words, dts, T)
        smp, ctl = emu_expand(em, iv, words, dts, off, T, packed=True)
        check_against_host(em, iv, dt, var, value, off, T, smp, ctl, full_lists=False)
        for s in (0, 2, 4):
            assert_bits(smp[s], np.repeat(iv[s][None, :], T, axis=0), "empty track")
            assert ctl[s].shape == (0, 2)


def test_scaled_columns_are_two_rounded_operations(edge):
    _, em = edge
    iv = np.array([[1, 3.0]])
    dt, var, bins, off = lists([[(2, 2, 3), (1, 2, 1), (1, 0, 0)]])
    words, dts = rows_packed(em, dt, var, bins, np.array([5, 999, 0]))
    value = decode(em, words, dts, 4)
    spec = ([2, 2, 1], [1.0, math.pi / 180.0, 1.68780972222222], [60.0, 1.0, 3.0])
    _, ctl = emu_expand(em, iv, words, dts, off, 4, packed=True, spec=spec, samples=False)
    xs = [3.0, value[0], value[1]]
    want = np.array([[t, x / 60.0, x * (math.pi / 180.0), (1.0 * 1.68780972222222) / 3.0] for t, x in zip((0, 2, 3), xs)])
    assert_bits(ctl[0], want, "scaled control columns")


def test_n_zero(edge):
    _, em = edge
    smp, ctl = emu_expand(em, np.zeros((0, 2)), np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint8),
                          np.zeros(1, dtype=np.int64), 5, packed=True)
    assert smp.shape == (0, 5, 2) and ctl == []


def test_n_zero_through_the_library(edge):
    path, _ = edge
    m = EncounterModel(path)
    for rows, dts in ((np.zeros(0, dtype=L.EVENT_DTYPE), None), (np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint8))):
        smp, ctl = m.expand_events_gpu(rows, np.zeros(1, dtype=np.int64), 5, np.zeros((2, 0)), dts=dts)
        assert smp.shape == (0, 5, 2) and ctl.rows.shape == (0, 2) and list(ctl.offsets) == [0]


# ---- refusals found on the device (here: the emulation's status word) ------------------------------------------------------
DEVICE_REFUSALS = {
    # (rows (dt, var, bin), offsets or None, packed, expected bit)
    "variable above n_initial": ([(1, 3, 1), (1, 0, 0)], None, False, BAD_VAR),
    "packed bin above r": ([(1, 2, 4), (1, 0, 0)], None, True, BAD_BIN),
    "packed bin above r of a '*' variable": ([(1, 1, 3), (1, 0, 0)], None, True, BAD_BIN),
    "decreasing offsets": ([(1, 2, 2), (1, 0, 0)], [0, 2, 1], False, BAD_OFFSETS),
    "negative offset": ([(1, 2, 2), (1, 0, 0)], [-1, 2, 2], True, BAD_OFFSETS),
    "offsets beyond the last": ([(1, 2, 2), (1, 0, 0)], [0, 3, 2], False, BAD_OFFSETS),
}


@pytest.mark.parametrize("case", sorted(DEVICE_REFUSALS))
def test_bad_lists_raise_their_status_bit(edge, case):
    _, em = edge
    rows, off, packed, bit = DEVICE_REFUSALS[case]
    dt, var, bins, off0 = lists([rows])
    off = off0 if off is None else np.asarray(off, dtype=np.int64)
    iv = np.ones((len(off) - 1, 2))
    if packed:
        words, dts = np.zeros(len(dt), np.uint32), (dt & 255).astype(np.uint8)
        words[:] = (np.where(var > 0, var, 0) << 27) | (np.maximum(bins - 1, 0) << 23)   # gord = var here: A, B are gated 1, 2
        emu_expand(em, iv, words, dts, off, 4, packed=True, status=bit)
    else:
        emu_expand(em, iv, rows_8byte(dt, var, bins, 1.0), None, off, 4, packed=False, status=bit)


def test_packed_ordinal_above_n_gated(edge):
    _, em = edge
    words = np.array([(3 << 27) | (1 << 23), 0], dtype=np.uint32)   # gord 3 of a model with 2 gated variables
    emu_expand(em, np.ones((1, 2)), words, np.array([1, 1], np.uint8), np.array([0, 2]), 4, packed=True, status=BAD_VAR)


# ---- refusals of the C ABI before any device work -----------------------------------------------------------------------
INITIAL_ONLY = EDGE_MODEL.split("# labels_transition")[0] + "# boundaries\n*\n*\n# resample_rates\n0 0\n"
BUF = np.zeros(1 << 12)
P = BUF.ctypes.data
OFF = np.zeros(5, dtype=np.int64)


def opts(mem=L.EMB_MEM_HOST):
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem = mem
    return o


def spec(n_cols=1, var=1, mul=1.0, div=1.0):
    s = L.ControlsSpec()
    s.n_cols = n_cols
    for j in range(8):
        s.vars[j], s.mul[j], s.div[j] = var, mul, div
    return s


def ex8(m, T, o=None, sp=None, capacity=0, controls=None):
    total = C.c_int64(-1)
    rc = L.lib().emb_track_events_expand(m._h, 4, T, P, P, OFF.ctypes.data, C.byref(o or opts()), sp and C.byref(sp), P,
                                         capacity, controls, P, C.byref(total))
    assert total.value == 0
    return rc


def exp(m, T, o=None, sp=None):
    return L.lib().emb_track_events_expand_packed(m._h, 4, T, P, P, P, OFF.ctypes.data, C.byref(o or opts()), sp and C.byref(sp),
                                                  P, 0, None, P, None)


HOST_REFUSALS = {
    "rows8/async": (lambda m, mi: ex8(m, 8, opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)), "EMB_MEM_ASYNC is not supported"),
    "packed/async": (lambda m, mi: exp(m, 8, opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)), "EMB_MEM_ASYNC is not supported"),
    "rows8/T < 1": (lambda m, mi: ex8(m, 0), "null or out-of-range argument"),
    "packed/T < 1": (lambda m, mi: exp(m, 0), "null or out-of-range argument"),
    "rows8/T > 65535": (lambda m, mi: ex8(m, 65536), "T <= 65535"),
    "packed/T > 1023": (lambda m, mi: exp(m, 1024), "T <= 1023"),
    "n_cols above EMB_MAX_DYN": (lambda m, mi: ex8(m, 8, sp=spec(9)), "n_cols must be 0..EMB_MAX_DYN"),
    "n_cols negative": (lambda m, mi: exp(m, 8, sp=spec(-1)), "n_cols must be 0..EMB_MAX_DYN"),
    "column variable 0": (lambda m, mi: ex8(m, 8, sp=spec(2, var=0)), "outside 1..n_initial"),
    "column variable above n_initial": (lambda m, mi: exp(m, 8, sp=spec(1, var=3)), "outside 1..n_initial"),
    "infinite mul": (lambda m, mi: ex8(m, 8, sp=spec(1, mul=math.inf)), "mul or div is not finite"),
    "NaN div": (lambda m, mi: exp(m, 8, sp=spec(3, div=math.nan)), "mul or div is not finite"),
    "rows8/no transition network": (lambda m, mi: ex8(mi, 8), "dynvar:empty"),
    "packed/no transition network": (lambda m, mi: exp(mi, 8, sp=spec(0)), "dynvar:empty"),
    "capacity without a buffer": (lambda m, mi: ex8(m, 8, capacity=5), "null or out-of-range argument"),
    "null rows": (lambda m, mi: L.lib().emb_track_events_expand(m._h, 4, 8, P, None, OFF.ctypes.data, C.byref(opts()), None, P,
                                                                0, None, P, None), "null or out-of-range argument"),
    "null dts": (lambda m, mi: L.lib().emb_track_events_expand_packed(m._h, 4, 8, P, P, None, OFF.ctypes.data, C.byref(opts()),
                                                                      None, P, 0, None, P, None), "null or out-of-range argument"),
}


@pytest.mark.parametrize("case", sorted(HOST_REFUSALS))
def test_host_refusals_launch_nothing(tmp_path, edge, case):
    path, _ = edge
    f = tmp_path / "initial_only.txt"
    f.write_text(INITIAL_ONLY)
    m, mi = EncounterModel(path), EncounterModel(str(f))
    call, message = HOST_REFUSALS[case]
    launches = L.lib().emb_launch_count()
    rc = call(m, mi)
    err = L.lib().emb_last_error().decode()
    assert (rc, message in err) == (L.EMB_E_ARG, True), (rc, err)
    assert L.lib().emb_launch_count() == launches


def test_python_wrapper_requires_init_values(edge):
    path, _ = edge
    m = EncounterModel(path)
    with pytest.raises(L.EmbError) as ei:
        m.expand_events_gpu(np.zeros(1, dtype=L.EVENT_DTYPE), np.zeros(2, dtype=np.int64), 4)
    assert ei.value.code == L.EMB_E_ARG and "init_values" in ei.value.message
