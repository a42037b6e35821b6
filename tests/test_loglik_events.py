"""CPU suite for scoring tracks given as event lists (emb_loglik_track_events[_packed]): the per-track routine of
emb_loglik_events.cuh, run on the host by the TEST-ONLY emulation in tests/emu/emu_loglik_events.cpp, against the independent
restatement in oracle/loglik_events.py and against the dense scoring (emu_loglik.cpp) of the same tracks expanded and tiled;
the refusals of the C ABI that need no device."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import cases
from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel, expand_events, tile
from helpers import ROOT
from oracle.em_read import em_read
from oracle import loglik as OL
from oracle import loglik_events as OE

# status bits of emb_loglik.cuh / emb_loglik_events.cuh
BAD_BIN, BAD_COL0, BAD_VAR, BAD_STATIC, BAD_OFFSETS = 1, 2, 4, 8, 16

_ll = None


def _lib():
    """Build (once per process, into a temporary directory: the tree may be read-only) and load both scoring emulations."""
    global _ll
    if _ll is not None:
        return _ll
    out = os.path.join(tempfile.mkdtemp(prefix="emb_loglik_events_emu_"), "libemb_loglik_events_emu.so")
    srcs = [os.path.join(ROOT, "tests", "emu", "emu_loglik.cpp"), os.path.join(ROOT, "tests", "emu", "emu_loglik_events.cpp"),
            os.path.join(ROOT, "em_model_manned_bayes_b200", "csrc", "emb_model.cpp")]
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared",
                    "-I", "/usr/local/cuda/include"] + srcs + ["-o", out], check=True)
    lib = C.CDLL(out)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.ll_last_error.restype = C.c_char_p
    lib.ll_model_load.argtypes = [C.c_char_p, C.c_int, C.POINTER(i32), i32, C.POINTER(vp)]
    lib.ll_model_free.argtypes = [vp]
    lib.ll_set_prior.argtypes = [vp, C.c_int, C.c_int, C.c_double]
    lib.ll_loglik_tracks.argtypes = [vp, i64, i32, vp, vp, i32, vp, vp]
    lib.lle_loglik_events.argtypes = [vp, i64, i32, vp, vp, vp, vp, i32, i32, vp, vp]
    _ll = lib
    return lib


class EmuModel:
    """A model loaded into the scoring emulation (tests only), with the library's view of it for the gated ordinals."""

    def __init__(self, path, idx_zero=(), overwrite=False):
        self.lib = _lib()
        self.h = C.c_void_p()
        idx = (C.c_int32 * max(1, len(idx_zero)))(*idx_zero)
        rc = self.lib.ll_model_load(path.encode(), int(overwrite), idx, len(idx_zero), C.byref(self.h))
        assert rc == 0, self.lib.ll_last_error()
        self.m = EncounterModel(path)

    def __del__(self):
        try:
            if self.h.value:
                self.lib.ll_model_free(self.h)
                self.h = C.c_void_p()
        except Exception:
            pass


def rows_8byte(dt, var, bins):
    ev = np.zeros(len(dt), dtype=L.EVENT_DTYPE)
    ev["dt"], ev["var"], ev["bin"] = dt, var, bins
    ev["value"] = 12.5                                 # ignored by the scoring
    return ev


def rows_packed(em, dt, var, bins):
    """the 5-byte rows of emb_sample_track_events_packed (frac 0) for the same (dt, var, bin) rows"""
    gord_of = {int(v): k + 1 for k, v in enumerate(em.m.gated_vars)}
    dt, var, bins = (np.asarray(a, dtype=np.int64) for a in (dt, var, bins))
    gord = np.array([gord_of[int(v)] if v > 0 else 0 for v in var], dtype=np.int64)
    words = (np.where(gord > 0, bins - 1, 0) << 23) | (gord << 27) | ((dt >> 8) << 30)
    return words.astype(np.uint32), (dt & 255).astype(np.uint8)


def emu_events(em, init_bins, dt, var, bins, offsets, T, correct_dbn=False, packed=False, status=0):
    """init_bins (n, n_initial) -> (initial, transition); asserts the status bits the call raises"""
    ib = np.ascontiguousarray(np.asarray(init_bins).T, dtype=np.int8)
    n = ib.shape[1]
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    if packed:
        rows, dts = rows_packed(em, dt, var, bins)
    else:
        rows, dts = rows_8byte(dt, var, bins), np.zeros(1, dtype=np.uint8)
    rows = rows if len(rows) else np.zeros(1, dtype=rows.dtype)
    init, trans = np.zeros(n), np.zeros(n)
    got = _lib().lle_loglik_events(em.h, n, T, ib.ctypes.data, rows.ctypes.data, dts.ctypes.data, off.ctypes.data, int(packed),
                                   int(correct_dbn), init.ctypes.data, trans.ctypes.data)
    assert got == status, "status %d, expected %d" % (got, status)
    return init, trans


def emu_dense(em, init_bins, dense, correct_dbn=False):
    """the dense scoring (emb_loglik_tracks) of (n, n_dyn, T) bins"""
    ib = np.ascontiguousarray(np.asarray(init_bins).T, dtype=np.int8)
    n, _, T = dense.shape
    bt = tile(np.asarray(dense, dtype=np.int8))
    init, trans = np.zeros(n), np.zeros(n)
    rc = _lib().ll_loglik_tracks(em.h, n, T, ib.ctypes.data, bt.ctypes.data, int(correct_dbn), init.ctypes.data, trans.ctypes.data)
    assert rc == 0, _lib().ll_last_error()
    return init, trans


def expanded(em, init_bins, dt, var, bins, offsets, T):
    """(n, n_dyn, T) dense bins of the lists, through the library's own expand_events"""
    init_bins = np.asarray(init_bins)
    if len(dt) == 0:                                   # (expand_events needs at least one row)
        full = np.repeat(init_bins[:, :, None], T, axis=2)
    else:
        full = expand_events(init_bins, dt, var, bins, offsets, T)
    return full[:, np.asarray(em.m.temporal_map)[:, 0] - 1, :].astype(np.int8)


def assert_same(got, want, rtol=1e-12):
    got, want = np.asarray(got), np.asarray(want)
    assert not np.isnan(got).any() and not np.isnan(want).any()
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf) and np.array_equal(got[inf], want[inf]), "-inf terms differ"
    assert np.all(np.abs(got[~inf] - want[~inf]) <= rtol * np.maximum(np.abs(want[~inf]), 1e-300)), \
        "max rel %g" % np.max(np.abs(got[~inf] - want[~inf]) / np.maximum(np.abs(want[~inf]), 1e-300))


def golden_rows(g):
    ev = g["events"]
    return ev[:, 0].astype(np.int64), ev[:, 1].astype(np.int64), g["event_bins"].astype(np.int64), g["event_offsets"]


@pytest.mark.parametrize("correct_dbn", [False, True], ids=["sampler_branch", "correct_dbn"])
@pytest.mark.parametrize("name", sorted(cases.TRACK_CASES))
def test_golden_lists_match_oracle_and_dense_scoring(model_paths, golden, name, correct_dbn):
    c, g = cases.TRACK_CASES[name], golden[name]
    path, ow = model_paths[c["model"]], c.get("overwrite", ())
    p = em_read(path, isOverwriteZeroBoundaries=bool(ow), idxZeroBoundaries=ow or (1, 2, 3))
    em = EmuModel(path, idx_zero=ow, overwrite=bool(ow))
    prior = 0
    if c.get("prior") == "dbe":
        for which in (0, 1):
            assert _lib().ll_set_prior(em.h, which, L.EMB_PRIOR_DBE, 0.0) == 0
        prior = "dbe"
    T, init_bins = c["T"], g["init_bins"]
    dt, var, bins, off = golden_rows(g)
    dense = expanded(em, init_bins, dt, var, bins, off, T)
    assert np.array_equal(dense, g["bins"]), "the golden lists do not expand to the golden dense bins"

    init, trans = emu_events(em, init_bins, dt, var, bins, off, T, correct_dbn)
    wi, wt = OE.loglik_track_events(p, init_bins, dt, var, bins, off, T, prior=prior, correct_dbn=correct_dbn)
    assert_same(init, wi)
    assert_same(trans, wt)
    di, dtr = emu_dense(em, init_bins, dense, correct_dbn)
    assert np.array_equal(init, di), "initial term differs from the dense scoring"
    if not OL.is_dynvar_depend(p) and not correct_dbn:
        assert np.array_equal(trans, dtr), "frozen transition term differs from the dense scoring"
    else:
        assert_same(trans, dtr)
    if len(em.m.gated_vars) <= 7 and T <= 1023:       # the packed format
        pi, pt = emu_events(em, init_bins, dt, var, bins, off, T, correct_dbn, packed=True)
        assert np.array_equal(pi, init) and np.array_equal(pt, trans), "packed rows score differently"


# ---- edge lists on a hand-made model ------------------------------------------------------------------------------------
# initial A (r=2) -> B (r=3); transition: B(t) -> B(t+1), A static.  Column A=2 of B is all zero (bin 1 with probability 1);
# transition column B(t)=3 is all zero, bin 3 of column B(t)=1 has weight 0.  B is resampled so that it is gated.
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
*
# resample_rates
0.1 0.1
"""


@pytest.fixture
def edge(tmp_path):
    f = tmp_path / "edge.txt"
    f.write_text(EDGE_MODEL)
    return str(f), EmuModel(str(f)), em_read(str(f))


def lists(tracks):
    """[[(dt, var, bin), ...] per track] -> dt, var, bin, offsets"""
    rows = [r for t in tracks for r in t]
    off = np.concatenate(([0], np.cumsum([len(t) for t in tracks]))).astype(np.int64)
    a = np.array(rows, dtype=np.int64).reshape(-1, 3)
    return a[:, 0], a[:, 1], a[:, 2], off


EDGE_LISTS = {
    # (init (A, B), rows (dt, var, bin), T)
    "several rows of one variable in one second": ((1, 1), [(2, 2, 2), (0, 2, 3), (0, 2, 1), (0, 2, 2), (3, 0, 0)], 5),
    "rows at column >= T": ((1, 1), [(1, 2, 2), (3, 2, 1), (1, 2, 3), (0, 0, 0)], 4),
    "sum dt < T": ((1, 2), [(1, 2, 1), (1, 2, 2)], 7),
    "closing row only": ((2, 1), [(6, 0, 0)], 6),
    "no rows": ((1, 1), [], 3),
    "T = 1": ((1, 2), [(1, 2, 1), (1, 0, 0)], 1),
    "zero-weight bin": ((1, 1), [(1, 2, 3), (2, 2, 1), (1, 0, 0)], 4),
    "zero-total column": ((1, 3), [(2, 2, 2), (2, 2, 1), (1, 0, 0)], 5),
    "column 0 rows": ((1, 2), [(0, 2, 3), (0, 2, 2), (0, 1, 1), (2, 2, 1), (2, 0, 0)], 4),
    "static resample rows": ((2, 1), [(1, 1, 2), (1, 2, 2), (0, 1, 2), (2, 0, 0)], 4),
    "change back within a second": ((1, 1), [(2, 2, 2), (0, 2, 1), (3, 0, 0)], 5),
}


@pytest.mark.parametrize("packed", [False, True], ids=["rows8", "packed"])
@pytest.mark.parametrize("correct_dbn", [False, True], ids=["frozen", "per_step"])
@pytest.mark.parametrize("case", sorted(EDGE_LISTS))
def test_edge_lists_match_oracle(edge, case, correct_dbn, packed):
    _, em, p = edge
    init, rows, T = EDGE_LISTS[case]
    ib = np.array([init], dtype=np.int8)
    dt, var, bins, off = lists([rows])
    i, t = emu_events(em, ib, dt, var, bins, off, T, correct_dbn, packed=packed)
    wi, wt = OE.loglik_track_events(p, ib, dt, var, bins, off, T, correct_dbn=correct_dbn)
    assert_same(i, wi)
    assert_same(t, wt)
    di, dtr = emu_dense(em, ib, expanded(em, ib, dt, var, bins, off, T), correct_dbn)
    assert np.array_equal(i, di)
    if correct_dbn:
        assert_same(t, dtr)
    else:
        assert np.array_equal(t, dtr)
    if T == 1:
        assert t[0] == 0.0


def test_edge_values(edge):
    _, em, p = edge
    ib = np.array([[1, 1], [1, 3]], dtype=np.int8)
    dt, var, bins, off = lists([[(1, 2, 3), (3, 0, 0)], [(1, 2, 1), (3, 0, 0)]])
    _, t = emu_events(em, ib, dt, var, bins, off, 4)
    assert t[0] == -math.inf                          # B 1 -> 3 has weight 0
    assert t[1] == 0.0                                # frozen in the empty column of B(0) = 3: bin 1 has probability 1
    _, t = emu_events(em, ib, dt, var, bins, off, 4, correct_dbn=True)
    assert t[1] == 2.0 * math.log(0.5)                # 3 -> 1 in the empty column, then 1 -> 1 twice as one product
    dt, var, bins, off = lists([[(1, 2, 2), (2, 2, 1), (1, 0, 0)]])
    _, t = emu_events(em, ib[:1], dt, var, bins, off, 6, correct_dbn=True)
    # B = 1, 2, 2, 1, 1, 1: one term per run of constant state, in time order -- 1 -> 2, then 2 -> 2 once, 2 -> 1, then
    # 1 -> 1 twice as one product
    want = 0.0
    for term in (math.log(5 / 10), 1.0 * math.log(2 / 6), math.log(1 / 6), 2.0 * math.log(5 / 10)):
        want += term
    assert t[0] == want


def test_ragged_batches_match_oracle(model_paths, golden):
    """many tracks, n not a multiple of 128, T shorter and longer than the lists: glider (frozen) and cor_v1 (per-step)"""
    for name in ("glider_n16_T120_seed6", "cor_v1_n12_T60_seed9"):
        c, g = cases.TRACK_CASES[name], golden[name]
        p, em = em_read(model_paths[c["model"]]), EmuModel(model_paths[c["model"]])
        dt, var, bins, off = golden_rows(g)
        rng = np.random.default_rng(len(name))
        pick = rng.integers(0, len(off) - 1, 133)
        parts = [np.arange(off[s], off[s + 1]) for s in pick]
        idx = np.concatenate(parts)
        noff = np.concatenate(([0], np.cumsum([len(q) for q in parts]))).astype(np.int64)
        for T in (1, 13, c["T"], c["T"] + 9):
            i, t = emu_events(em, g["init_bins"][pick], dt[idx], var[idx], bins[idx], noff, T)
            wi, wt = OE.loglik_track_events(p, g["init_bins"][pick], dt[idx], var[idx], bins[idx], noff, T)
            assert_same(i, wi)
            assert_same(t, wt)


def test_n_zero(edge):
    _, em, _ = edge
    i, t = emu_events(em, np.zeros((0, 2), dtype=np.int8), [], [], [], np.zeros(1, dtype=np.int64), 5)
    assert i.shape == (0,) and t.shape == (0,)


def test_n_zero_through_the_library(edge):
    path, _, _ = edge
    m = EncounterModel(path)
    ev = np.zeros(0, dtype=L.EVENT_DTYPE)
    i, t = m.loglik_events(ev, np.zeros(1, dtype=np.int64), 5, np.zeros((2, 0), dtype=np.int8))
    assert i.shape == (0,) and t.shape == (0,)
    i, t = m.loglik_events(np.zeros(0, dtype=np.uint32), np.zeros(1, dtype=np.int64), 5, np.zeros((2, 0), dtype=np.int8),
                           dts=np.zeros(0, dtype=np.uint8))
    assert i.shape == (0,) and t.shape == (0,)


# ---- refusals found on the device (here: the emulation's status word) ------------------------------------------------------
DEVICE_REFUSALS = {
    # (init (A, B), rows, offsets or None, packed, expected bit)
    "bin above r": ((1, 1), [(1, 2, 4), (1, 0, 0)], None, False, BAD_BIN),
    "bin 0": ((1, 1), [(1, 2, 0), (1, 0, 0)], None, False, BAD_BIN),
    "static bin above r": ((1, 1), [(1, 1, 3), (1, 0, 0)], None, False, BAD_BIN),
    "packed bin above r": ((1, 1), [(1, 2, 4), (1, 0, 0)], None, True, BAD_BIN),
    "variable above n_initial": ((1, 1), [(1, 3, 1), (1, 0, 0)], None, False, BAD_VAR),
    "static bin changes": ((1, 1), [(1, 1, 2), (1, 0, 0)], None, False, BAD_STATIC),
    "static bin changes after T": ((1, 1), [(9, 1, 2)], None, False, BAD_STATIC),
    "column 0 differs": ((1, 1), [(0, 2, 2), (2, 0, 0)], None, False, BAD_COL0),
    "packed column 0 differs": ((1, 1), [(0, 2, 2), (2, 0, 0)], None, True, BAD_COL0),
    "decreasing offsets": ((1, 1), [(1, 2, 2), (1, 0, 0)], [0, 2, 1], False, BAD_OFFSETS),
    "negative offset": ((1, 1), [(1, 2, 2), (1, 0, 0)], [-1, 2, 2], False, BAD_OFFSETS),
}


@pytest.mark.parametrize("correct_dbn", [False, True], ids=["frozen", "per_step"])
@pytest.mark.parametrize("case", sorted(DEVICE_REFUSALS))
def test_bad_lists_raise_their_status_bit(edge, case, correct_dbn):
    _, em, _ = edge
    init, rows, off, packed, bit = DEVICE_REFUSALS[case]
    dt, var, bins, off0 = lists([rows])
    if off is None:
        ib, off = np.array([init], dtype=np.int8), off0
    else:
        ib = np.array([init, init], dtype=np.int8)
    emu_events(em, ib, dt, var, bins, np.asarray(off, dtype=np.int64), 4, correct_dbn, packed=packed, status=bit)


def test_packed_ordinal_above_n_gated(edge):
    _, em, _ = edge
    words = np.array([(3 << 27) | (1 << 23) | 0, 0], dtype=np.uint32)   # gord 3 of a model with 2 gated variables
    dts = np.array([1, 1], dtype=np.uint8)
    ib = np.ascontiguousarray(np.array([[1, 1]], dtype=np.int8).T)
    off = np.array([0, 2], dtype=np.int64)
    init, trans = np.zeros(1), np.zeros(1)
    st = _lib().lle_loglik_events(em.h, 1, 4, ib.ctypes.data, words.ctypes.data, dts.ctypes.data, off.ctypes.data, 1, 0,
                                  init.ctypes.data, trans.ctypes.data)
    assert st == BAD_VAR


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


def ev8(m, T, o=None):
    return L.lib().emb_loglik_track_events(m._h, 4, T, P, P, OFF.ctypes.data, C.byref(o or opts()), P, P)


def evp(m, T, o=None):
    return L.lib().emb_loglik_track_events_packed(m._h, 4, T, P, P, P, OFF.ctypes.data, C.byref(o or opts()), P, P)


HOST_REFUSALS = {
    "rows8/async": (lambda m, mi: ev8(m, 8, opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)), "EMB_MEM_ASYNC is not supported"),
    "packed/async": (lambda m, mi: evp(m, 8, opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)), "EMB_MEM_ASYNC is not supported"),
    "rows8/no transition network": (lambda m, mi: ev8(mi, 8), "dynvar:empty"),
    "packed/no transition network": (lambda m, mi: evp(mi, 8), "dynvar:empty"),
    "rows8/T < 1": (lambda m, mi: ev8(m, 0), "null or out-of-range argument"),
    "packed/T < 1": (lambda m, mi: evp(m, 0), "null or out-of-range argument"),
    "rows8/T > 65535": (lambda m, mi: ev8(m, 65536), "T <= 65535"),
    "packed/T > 1023": (lambda m, mi: evp(m, 1024), "T <= 1023"),
    "rows8/null rows": (lambda m, mi: L.lib().emb_loglik_track_events(m._h, 4, 8, P, None, OFF.ctypes.data, C.byref(opts()), P, P),
                        "null or out-of-range argument"),
    "packed/null dts": (lambda m, mi: L.lib().emb_loglik_track_events_packed(m._h, 4, 8, P, P, None, OFF.ctypes.data,
                                                                              C.byref(opts()), P, P),
                        "null or out-of-range argument"),
}


@pytest.mark.parametrize("case", sorted(HOST_REFUSALS))
def test_host_refusals_launch_nothing(tmp_path, edge, case):
    path, _, _ = edge
    f = tmp_path / "initial_only.txt"
    f.write_text(INITIAL_ONLY)
    m, mi = EncounterModel(path), EncounterModel(str(f))
    call, message = HOST_REFUSALS[case]
    launches = L.lib().emb_launch_count()
    rc = call(m, mi)
    err = L.lib().emb_last_error().decode()
    assert (rc, message in err) == (L.EMB_E_ARG, True), (rc, err)
    assert L.lib().emb_launch_count() == launches


def test_python_wrapper_requires_init_bins(edge):
    path, _, _ = edge
    m = EncounterModel(path)
    with pytest.raises(L.EmbError) as ei:
        m.loglik_events(np.zeros(1, dtype=L.EVENT_DTYPE), np.zeros(2, dtype=np.int64), 4)
    assert ei.value.code == L.EMB_E_ARG and "init_bins" in ei.value.message
