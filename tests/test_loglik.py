"""CPU suite for the log-likelihood entry points: the scoring routines of emb_loglik.cuh, run on the host by the TEST-ONLY
emulation in tests/emu/emu_loglik.cpp, against the independent restatement in oracle/loglik.py; the packed log tables against numpy; the
argument checks of the C ABI that need no device."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import cases
from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel, tile
from helpers import ROOT
from oracle.em_read import em_read
from oracle import loglik as OL

_ll = None


def _lib():
    """Build (once per process, into a temporary directory: the tree may be read-only) and load tests/emu/emu_loglik.cpp."""
    global _ll
    if _ll is not None:
        return _ll
    out = os.path.join(tempfile.mkdtemp(prefix="emb_loglik_emu_"), "libemb_loglik_emu.so")
    srcs = [os.path.join(ROOT, "tests", "emu", "emu_loglik.cpp"),
            os.path.join(ROOT, "em_model_manned_bayes_b200", "csrc", "emb_model.cpp")]
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared",
                    "-I", "/usr/local/cuda/include"] + srcs + ["-o", out], check=True)
    lib = C.CDLL(out)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.ll_last_error.restype = C.c_char_p
    lib.ll_model_load.argtypes = [C.c_char_p, C.c_int, C.POINTER(i32), i32, C.POINTER(vp)]
    lib.ll_model_free.argtypes = [vp]
    lib.ll_set_prior.argtypes = [vp, C.c_int, C.c_int, C.c_double]
    lib.ll_loglik_initial.argtypes = [vp, i64, vp, vp, vp]
    lib.ll_loglik_tracks.argtypes = [vp, i64, i32, vp, vp, i32, vp, vp]
    lib.ll_model_get_logp.argtypes = [vp, C.c_int, vp, i64]
    lib.ll_model_get_logp.restype = i64
    _ll = lib
    return lib


def _check(rc):
    if rc:
        raise L.EmbError(rc, _lib().ll_last_error().decode())


class EmuModel:
    """A model loaded into the scoring emulation (tests only)."""

    def __init__(self, path, idx_zero=(), overwrite=False):
        self.lib = _lib()
        self.h = C.c_void_p()
        idx = (C.c_int32 * max(1, len(idx_zero)))(*idx_zero)
        _check(self.lib.ll_model_load(path.encode(), int(overwrite), idx, len(idx_zero), C.byref(self.h)))

    def __del__(self):
        try:
            if self.h.value:
                self.lib.ll_model_free(self.h)
                self.h = C.c_void_p()
        except Exception:
            pass

    def set_prior(self, which, kind, value):
        _check(self.lib.ll_set_prior(self.h, which, kind, value))


def emu_initial(em, bins):
    """bins (n, n_initial) -> (total, per_var (n, n_initial))"""
    b = np.ascontiguousarray(np.asarray(bins).T, dtype=np.int8)
    n = b.shape[1]
    total = np.zeros(n)
    pv = np.zeros(b.shape)
    _check(_lib().ll_loglik_initial(em.h, n, b.ctypes.data, total.ctypes.data, pv.ctypes.data))
    return total, pv.T


def emu_tracks(em, init_bins, bins, correct_dbn=False, tiled=None):
    """init_bins (n, n_initial), bins (n, n_dyn, T) -> (initial, transition)"""
    ib = np.ascontiguousarray(np.asarray(init_bins).T, dtype=np.int8)
    n, _, T = bins.shape
    bt = tile(np.asarray(bins, dtype=np.int8)) if tiled is None else tiled
    init, trans = np.zeros(n), np.zeros(n)
    _check(_lib().ll_loglik_tracks(em.h, n, T, ib.ctypes.data, bt.ctypes.data, int(correct_dbn), init.ctypes.data,
                                   trans.ctypes.data))
    return init, trans


def assert_same(got, want, rtol=1e-12):
    got, want = np.asarray(got), np.asarray(want)
    assert not np.isnan(got).any() and not np.isnan(want).any()
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf) and np.array_equal(got[inf], want[inf]), "-inf terms differ"
    assert np.all(np.abs(got[~inf] - want[~inf]) <= rtol * np.maximum(np.abs(want[~inf]), 1e-300)), \
        "max rel %g" % np.max(np.abs(got[~inf] - want[~inf]) / np.maximum(np.abs(want[~inf]), 1e-300))


def _emu_model(model_paths, c):
    path = model_paths[c["model"]]
    ow = c.get("overwrite", ())
    p = em_read(path, isOverwriteZeroBoundaries=bool(ow), idxZeroBoundaries=ow or (1, 2, 3))
    em = EmuModel(path, idx_zero=ow, overwrite=bool(ow))
    prior = 0
    if c.get("prior") == "dbe":
        em.set_prior(0, L.EMB_PRIOR_DBE, 0.0)
        em.set_prior(1, L.EMB_PRIOR_DBE, 0.0)
        prior = "dbe"
    return p, em, prior


@pytest.mark.parametrize("correct_dbn", [False, True], ids=["sampler_branch", "correct_dbn"])
@pytest.mark.parametrize("name", sorted(cases.TRACK_CASES))
def test_tracks_match_oracle(model_paths, golden, name, correct_dbn):
    c, g = cases.TRACK_CASES[name], golden[name]
    p, em, prior = _emu_model(model_paths, c)
    init, trans = emu_tracks(em, g["init_bins"], g["bins"], correct_dbn)
    wi, wt = OL.loglik_tracks(p, g["init_bins"], g["bins"], prior=prior, correct_dbn=correct_dbn)
    assert_same(init, wi)
    assert_same(trans, wt)
    # the tracks were sampled from this model (rejection only truncates): every sampled transition has positive probability
    # on the branch that drew it
    if not correct_dbn:
        assert np.isfinite(trans).all() and np.isfinite(init).all()
    assert np.array_equal(init, emu_initial(em, g["init_bins"])[0]), "track initial term != emb_loglik_initial"


@pytest.mark.parametrize("name", sorted(cases.INITIAL_CASES) + sorted(cases.TERMINAL_CASES))
def test_initial_matches_oracle(model_paths, golden, name):
    c = {**cases.INITIAL_CASES, **cases.TERMINAL_CASES}[name]
    p, em, prior = _emu_model(model_paths, c)
    bins = golden[name]["bins"]
    total, pv = emu_initial(em, bins)
    wt, wpv = OL.loglik_initial(p, bins, prior)
    assert_same(total, wt)
    assert_same(pv, wpv)
    assert np.isfinite(total).all()


def _expected_logp(tables):
    """numpy/libm log(w/W) of every column, padded to rp = 4*ceil(r/4) slots with -inf, in packing order"""
    out = []
    for w in tables:
        r, q = w.shape
        rp = (r + 3) // 4 * 4
        for j in range(q):
            col = w[:, j]
            W = float(np.cumsum(col)[-1])                                   # sequential, as select_random.m:17
            if not W > 0:
                v = [0.0] + [-math.inf] * (r - 1)
            else:
                v = [math.log(float(x) / W) if x > 0 else -math.inf for x in col]
            out.extend(v + [-math.inf] * (rp - r))
    return np.array(out)


@pytest.mark.parametrize("prior", [0, "dbe", 2.5])
@pytest.mark.parametrize("model", ["glider_v1", "cor_v1", "balloon_v1", "uncor_allcode_fwsingle_v1"])
def test_logp_tables_are_log_of_normalised_weights(model_paths, model, prior):
    m = EncounterModel(model_paths[model])                                  # the tables as emb_model_get_N returns them
    em = EmuModel(model_paths[model])
    if prior != 0:
        m.prior = prior
        kind, v = (L.EMB_PRIOR_DBE, 0.0) if prior == "dbe" else (L.EMB_PRIOR_CONSTANT, float(prior))
        em.set_prior(0, kind, v)
        em.set_prior(1, kind, v)

    def weights(N):
        r, q = N.shape
        return N + (1.0 / (r * q) if prior == "dbe" else float(prior))
    lib = _lib()
    for which in (0, 1):
        if which == 0:
            tabs = [weights(t) for t in m.N_initial]
        else:
            tabs = [weights(m.N_transition[int(v) - 1]) for v in m.temporal_map[:, 1]]   # packed in temporal_map order
        k = lib.ll_model_get_logp(em.h, which, None, 0)
        got = np.zeros(k)
        lib.ll_model_get_logp(em.h, which, got.ctypes.data, k)
        want = _expected_logp(tabs)
        assert got.shape == want.shape
        assert np.array_equal(got, want), "logp table %d differs" % which


# ---- edge cases on a hand-made model -------------------------------------------------------------------------------------
# initial A (r=2) -> B (r=3); transition: B(t) -> B(t+1).  Column A=2 of B is all zero (bin 1 with probability 1);
# bin 2 of column A=1 has weight 0; transition column B(t)=3 is all zero, bin 3 of column B(t)=1 has weight 0.
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
0 0
"""
INITIAL_ONLY = EDGE_MODEL.split("# labels_transition")[0] + "# boundaries\n*\n*\n# resample_rates\n0 0\n"


@pytest.fixture
def edge(tmp_path):
    f = tmp_path / "edge.txt"
    f.write_text(EDGE_MODEL)
    return str(f)


def test_zero_total_column_and_zero_weight_bin(edge):
    em = EmuModel(edge)
    p = em_read(edge)
    # (A, B): A=2 column is empty -> B=1 has log-prob 0, B=2,3 -inf; A=1: B=2 has weight 0 -> -inf
    bins = np.array([[2, 1], [2, 2], [2, 3], [1, 1], [1, 2], [1, 3]], dtype=np.int8)
    total, pv = emu_initial(em, bins)
    lA = [math.log(3 / 4), math.log(1 / 4)]
    want_B = [math.log(1 / 5), -math.inf, math.log(4 / 5)]
    assert pv[0, 1] == 0.0 and pv[1, 1] == -math.inf and pv[2, 1] == -math.inf
    assert [pv[3 + k, 1] for k in range(3)] == want_B
    assert list(pv[:, 0]) == [lA[1]] * 3 + [lA[0]] * 3
    assert not np.isnan(total).any() and not np.isnan(pv).any()
    assert_same(total, OL.loglik_initial(p, bins)[0])
    # transitions: B(t)=1 -> {5,5,0}: 3 is -inf; B(t)=3 -> empty column: only 1 (log 0)
    init = np.array([[1, 1], [1, 1], [1, 3], [1, 3]], dtype=np.int8)
    tracks = np.array([[[1, 2, 2, 1, 1]], [[1, 3, 1, 1, 1]], [[3, 1, 1, 1, 1]], [[3, 2, 2, 2, 2]]], dtype=np.int8)   # T = 5
    i, t = emu_tracks(em, init, tracks)
    assert not np.isnan(t).any() and not np.isnan(i).any()
    wi, wt = OL.loglik_tracks(p, init, tracks)
    assert_same(i, wi)
    assert_same(t, wt)
    assert t[1] == -math.inf and t[3] == -math.inf and np.isfinite(t[0])
    assert t[0] == 4 * math.log(0.5)
    assert t[2] == 0.0                                # frozen in the empty column of B(0) = 3: bin 1 has probability 1


def test_edge_track_frozen_column_is_column_zero(edge):
    em = EmuModel(edge)
    init = np.array([[1, 3]], dtype=np.int8)
    trk = np.array([[[3, 1, 1, 1, 1]]], dtype=np.int8)
    _, t = emu_tracks(em, init, trk)
    assert t[0] == 0.0                                # every step scored in the (empty) column of B(t) = 3
    _, t2 = emu_tracks(em, init, trk, correct_dbn=True)
    # per-step: step 1 from B=3 (empty column, bin 1: 0), then three steps 1 -> 1 (log 0.5 each)
    assert t2[0] == 3 * math.log(0.5)


@pytest.mark.parametrize("n,T", [(1, 1), (5, 2), (129, 7), (300, 33)])
def test_ragged_sizes_match_oracle(model_paths, golden, n, T):
    """n not a multiple of 128 and T not a multiple of 4: tracks resampled from the golden glider case (the branch of
    their parents follows the model, so any bins in range are valid input)."""
    c, g = cases.TRACK_CASES["glider_n16_T120_seed6"], golden["glider_n16_T120_seed6"]
    p, em, prior = _emu_model(model_paths, c)
    rng = np.random.default_rng(n * 1000 + T)
    pick = rng.integers(0, g["bins"].shape[0], n)
    init, bins = g["init_bins"][pick], g["bins"][pick][:, :, :T]
    tiled = tile(bins)
    tiled[tiled == 0] = 99                            # padding seconds / tracks must be ignored
    i, t = emu_tracks(em, init, bins, tiled=tiled)
    wi, wt = OL.loglik_tracks(p, init, bins)
    assert_same(i, wi)
    assert_same(t, wt)
    if T == 1:
        assert np.all(t == 0.0)


def test_n_zero(edge):
    em = EmuModel(edge)
    total, _ = emu_initial(em, np.zeros((0, 2), dtype=np.int8))
    assert total.shape == (0,)
    i, t = emu_tracks(em, np.zeros((0, 2), dtype=np.int8), np.zeros((0, 1, 5), dtype=np.int8))
    assert i.shape == (0,) and t.shape == (0,)


def test_n_zero_through_the_library(model_paths):
    """n = 0 returns before any device is touched"""
    m = EncounterModel(model_paths["glider_v1"])
    assert m.loglik_initial(np.zeros((0, m.n_initial), dtype=np.int8)).shape == (0,)
    i, t = m.loglik_tracks(np.zeros((m.n_initial, 0), dtype=np.int8), np.zeros(0, dtype=np.int8), 10)
    assert i.shape == (0,) and t.shape == (0,)


def test_bad_bins_are_refused(edge):
    em = EmuModel(edge)
    for bad in ([[3, 1]], [[1, 4]], [[0, 1]], [[1, -1]]):
        with pytest.raises(L.EmbError) as ei:
            emu_initial(em, np.array(bad, dtype=np.int8))
        assert ei.value.code == L.EMB_E_ARG and "outside 1..r" in ei.value.message
    init = np.array([[1, 1]], dtype=np.int8)
    with pytest.raises(L.EmbError) as ei:
        emu_tracks(em, init, np.array([[[1, 2, 4, 1, 1]]], dtype=np.int8))
    assert ei.value.code == L.EMB_E_ARG and "outside 1..r" in ei.value.message
    with pytest.raises(L.EmbError) as ei:
        emu_tracks(em, init, np.array([[[1, 2, 2, 1, 0]]], dtype=np.int8), correct_dbn=True)
    assert ei.value.code == L.EMB_E_ARG
    with pytest.raises(L.EmbError) as ei:
        emu_tracks(em, init, np.array([[[2, 2, 2, 1, 1]]], dtype=np.int8))
    assert ei.value.code == L.EMB_E_ARG and "column 0" in ei.value.message


def test_initial_only_model_has_no_track_likelihood(tmp_path, edge):
    f = tmp_path / "initial_only.txt"
    f.write_text(INITIAL_ONLY)
    em = EmuModel(str(f))
    with pytest.raises(L.EmbError) as ei:
        emu_tracks(em, np.ones((1, 2), dtype=np.int8), np.ones((1, 1, 4), dtype=np.int8))
    assert ei.value.code == L.EMB_E_ARG and "dynvar:empty" in ei.value.message
    m = EncounterModel(str(f))                        # the C ABI refuses before touching a device
    with pytest.raises(L.EmbError) as ei:
        m.loglik_tracks(np.ones((2, 3), dtype=np.int8), np.zeros(0, dtype=np.int8), 4)
    assert ei.value.code == L.EMB_E_ARG and "dynvar:empty" in ei.value.message


def test_async_is_refused(model_paths):
    m = EncounterModel(model_paths["glider_v1"])
    o = m._opts()
    o.mem = L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC
    out = np.zeros(1)
    b = np.ones((m.n_initial, 1), dtype=np.int8)
    rc = L.lib().emb_loglik_initial(m._h, 1, b.ctypes.data, C.byref(o), out.ctypes.data, None)
    assert rc == L.EMB_E_ARG
