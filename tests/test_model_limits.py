"""CPU suite for models at the compiled limits (tests/limit_models.py): each case first proves, from the loaded model alone, that
it reaches the branch it was made for; then the plain-C oracle against the Python oracle, and the host emulation of the device
code (tests/emu) against both -- sampling, event rows, scoring, expansion and formatting -- at shapes no shipped model has;
the array constructor; and the refusals one past each limit.  test_gpu_model_limits.py runs the same cases on the device."""
import numpy as np
import pytest

import helpers as H
import limit_models as LM
import test_events_expand as TX
import test_loglik as TL
import test_loglik_events as TE
from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel, tile
from oracle import loglik as OL
from oracle import loglik_events as OE
from oracle.c_oracle import COracle
from oracle.drivers import dbn_tracks, initial_sample
from oracle.em_read import em_read
from oracle.uniforms import KeyedPhilox
from test_format import emu_text, rows_transition

INIT_SHAPES = (2, 5, 6, 7, 9, 15)          # emb_initial.cuh: EMB_INIT_SHAPES
DBN = sorted(k for k in LM.CASES if k not in ("init15_wide", "staging_under", "staging_over"))
TWINS = ("fast_shape_twin", "fast_shape_twin_step")
EVENTS = [k for k in DBN if k not in ("wide_frozen", "hist64")]   # event rows need gated variables of <= 16 bins
FIRST = 2 ** 32 - 17                      # the tracks of every CPU case straddle sample 2^32


@pytest.fixture(scope="module")
def paths(tmp_path_factory):
    return LM.write_all(str(tmp_path_factory.mktemp("limit_models")))


def layout(p):
    """0-based dynamic variables (temporal_map order) and time-varying variables (the value rows of emb_sample_tracks)"""
    dyn = [int(v) - 1 for v in np.asarray(p.temporal_map)[:, 0]]
    rates = np.asarray(p.resample_rates)
    return dyn, sorted(set(dyn) | {i for i in range(p.n_initial) if rates[i] > 0})


# ---- what each case reaches, from the loaded model ------------------------------------------------------------------------
def frozen_scoring_block(m):
    """emb_kernels.cu: loglik_frozen_block -- (threads per block, bytes of dynamic shared memory)"""
    per_thread = 4 * int(sum(m.r_initial[int(v) - 1] for v in m.temporal_map[:, 0]))
    block = 128
    while block > 32 and per_thread * block > 96 * 1024:
        block //= 2
    return block, per_thread * block


def initial_table_bytes(m):
    """(bytes of the padded shared-memory table of k_initial_fast, bytes of the fp64 table of k_loglik_initial)"""
    cols = sum(int(np.prod(m.r_initial[m.G_initial[:, i]])) for i in range(m.n_initial))
    slots = len(m.packed(0))
    return 4 * (slots + 4 * cols), 8 * slots


def initial_is_fast(m):
    return m.n_initial in INIT_SHAPES and m.order_initial == list(range(1, m.n_initial + 1))


def gate_position_of_dyn(m):
    return [m.gated_vars.index(int(v)) for v in m.temporal_map[:, 0]]


def dyn_order(m):
    """order_transition restricted to the dynamic (t+1) nodes, as dynamic ordinals (DevModel::order_dyn)"""
    t1 = [int(v) for v in m.temporal_map[:, 1]]
    return [t1.index(v) for v in m.order_transition if v in t1]


def assert_branch(name, m):
    """The branch `name` is made for, asserted from the library's view of the model; a model that silently fell back to a
    shape the shipped models already cover fails here."""
    r, dyn_r = m.r_initial, [int(m.r_initial[int(v) - 1]) for v in m.temporal_map[:, 0]]
    gated_r = [int(r[v - 1]) for v in m.gated_vars]
    if name == "wide_frozen":
        assert (m.n_initial, m.n_dyn, m.n_gated) == (L.EMB_MAX_VARS, L.EMB_MAX_DYN, L.EMB_MAX_GATED)
        assert not m.is_dynvar_depend and m.order_initial != list(range(1, 25))
        assert min(dyn_r) >= 100 and max(r) == 127
        block, smem = frozen_scoring_block(m)
        assert block < 128 and smem > 96 * 1024, (block, smem)
        assert max(gated_r) > 16                                  # no event rows
    elif name == "deep_step":
        assert m.is_dynvar_depend and m.n_dyn == 8 and 8 <= m.n_gated <= 15 and max(gated_r) <= 16
        pos = gate_position_of_dyn(m)
        assert pos != list(range(m.n_gated - m.n_dyn, m.n_gated)), "gated list ends with the dynamic variables"
        assert max(pos) < m.n_gated - 1, "no resampled variable after a dynamic one"
        assert dyn_order(m) != list(range(8))
        assert int(m.G_transition.sum(axis=0).max()) == L.EMB_MAX_PARENTS
    elif name == "init15_wide":
        assert m.n_initial == 15 and m.n_transition == 0 and initial_is_fast(m)
        assert int(r.sum()) > 256 and max(r) == 127              # fp32 entries from global memory; a 128-slot column
    elif name == "hist64":
        assert max(r) == 64 and 64 in dyn_r
    elif name in ("staging_under", "staging_over"):
        assert initial_is_fast(m) and max(r) <= 4
        staged, logp = initial_table_bytes(m)
        assert staged == logp
        assert (staged <= 96 * 1024) == (name == "staging_under") and abs(staged - 96 * 1024) <= 32, staged
    elif name in TWINS:
        assert dyn_r == [5, 7, 7] and m.n_gated == 3 and m.is_dynvar_depend == (name == "fast_shape_twin_step")
        if m.is_dynvar_depend:
            assert dyn_order(m) == [1, 2, 0]
    else:
        raise AssertionError(name)


@pytest.mark.parametrize("name", sorted(LM.CASES))
def test_case_reaches_its_branch(paths, name):
    m = EncounterModel(paths[name])
    assert_branch(name, m)
    if name == "wide_frozen":
        with pytest.raises(L.EmbError) as ei:
            m.sample_tracks(4, 8, hist_initial=np.zeros((m.n_initial, 64), np.uint64))
        assert ei.value.code == L.EMB_E_LIMIT and "hold 64 bins" in ei.value.message
        with pytest.raises(L.EmbError) as ei:
            m.sample_events(4, 8)
        assert ei.value.code == L.EMB_E_LIMIT and "<= 16 bins" in ei.value.message
    if name == "deep_step":
        with pytest.raises(L.EmbError) as ei:
            m.sample_events_packed(4, 8)
        assert ei.value.code == L.EMB_E_LIMIT and "<= 7 time-varying variables" in ei.value.message


def test_histograms_refused_one_bin_past_the_stride(paths):
    m = EncounterModel(paths["hist65"])
    assert max(m.r_initial) == 65
    with pytest.raises(L.EmbError) as ei:
        m.sample_tracks(4, 8, hist_transition=np.zeros((m.n_dyn, 64), np.uint64))
    assert ei.value.code == L.EMB_E_LIMIT and "hold 64 bins" in ei.value.message


# ---- the two oracles -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(LM.CASES))
def test_c_oracle_equals_python_oracle(paths, name):
    p = em_read(paths[name])
    if not p.n_transition:
        n = 40
        ref = COracle(p).sample_initial(n, seed=3, first_sample=FIRST, threads=0)
        assert ref["rc"] == 0
        S, V = initial_sample(p, n, KeyedPhilox(3), first_sample=FIRST)
        assert np.array_equal(ref["bins"], S.astype(np.int8))
        assert np.all(np.abs(ref["values"] - V) <= 1e-12 * np.abs(V))
        return
    n, T = 6, 14
    ref = COracle(p).sample_tracks(n, T, seed=3, first_sample=FIRST, threads=0)
    assert ref["rc"] == 0
    for s, want in enumerate(dbn_tracks(p, n, T, KeyedPhilox(3), first_sample=FIRST)):
        assert np.array_equal(ref["init_bins"][s], want.initial_bins.astype(np.int8)), s
        assert np.array_equal(ref["sample_bins"][s], want.sample_bins.astype(np.int8)), s
        assert np.all(np.abs(ref["samples"][s] - want.samples) <= 1e-12 * np.abs(want.samples)), s
        assert np.all(np.abs(ref["init_values"][s] - want.samples[:, 0]) <= 1e-12 * np.abs(want.samples[:, 0])), s
        assert ref["attempts"][s] == 1 and ref["n_events"][s] == len(want.events), s


# ---- host emulation of the device code against the oracles ----------------------------------------------------------------
def emu_tracks(path, p, n, T, seed, first, fast, hist=False):
    """(emulated dense tracks, whether the specialised kernel ran)"""
    dyn, tv = layout(p)
    lib = H.emu_lib()
    lib.emu_use_fast(fast)
    try:
        got = H.EmuModel(path).sample_tracks(p.n_initial, len(dyn), len(tv), n, T, seed, first, H.EmuModel.opts(p.n_initial),
                                             hist=hist)
        return got, lib.emu_last_fast()
    finally:
        lib.emu_use_fast(0)


def check_tracks(got, ref, p, rtol=1e-6):
    """dense tracks (emb_sample_tracks layout) against a C-oracle result: bins, attempts, initial values exact"""
    dyn, tv = layout(p)
    assert np.array_equal(np.asarray(got["init_bins"]), ref["init_bins"]), "initial bins differ"
    assert np.array_equal(np.asarray(got["init_values"]), ref["init_values"]), "initial values differ"
    assert np.array_equal(np.asarray(got["attempts"]).astype(np.int64), ref["attempts"].astype(np.int64)), "attempts differ"
    assert np.array_equal(np.asarray(got["bins"]), ref["sample_bins"][:, dyn, :]), "track bins differ"
    want = ref["samples"][:, tv, :]
    gv = np.asarray(got["values"], dtype=np.float64)
    assert np.all(np.abs(gv - want) <= rtol * np.abs(want)), "track values differ by more than 1e-6 relative"


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "default"])
@pytest.mark.parametrize("name", DBN)
def test_emu_tracks_equal_c_oracle(paths, name, fast):
    p = em_read(paths[name])
    n, T = 48, 30
    ref = COracle(p).sample_tracks(n, T, seed=7, first_sample=FIRST, threads=0)
    assert ref["rc"] == 0
    got, used_fast = emu_tracks(paths[name], p, n, T, 7, FIRST, fast)
    assert used_fast == (fast and name in TWINS), "specialised kernel taken: %d" % used_fast
    check_tracks(got, ref, p)


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "default"])
@pytest.mark.parametrize("name", sorted(LM.CASES))
def test_emu_initial_equals_c_oracle(paths, name, fast):
    p = em_read(paths[name])
    n = 203
    ref = COracle(p).sample_initial(n, seed=9, first_sample=FIRST + 2, threads=0)
    lib = H.emu_lib()
    lib.emu_use_fast(fast)
    try:
        bins, vals, att = H.EmuModel(paths[name]).sample_initial(p.n_initial, n, 9, FIRST + 2, H.EmuModel.opts(p.n_initial))
        used_fast = lib.emu_last_fast()
    finally:
        lib.emu_use_fast(0)
    assert used_fast == (fast and initial_is_fast(EncounterModel(paths[name])))
    assert np.array_equal(bins, ref["bins"]) and np.array_equal(vals, ref["values"]) and np.all(att == 1)


def test_emu_histograms_at_the_stride(paths):
    p = em_read(paths["hist64"])
    n, T = 300, 25
    got, _ = emu_tracks(paths["hist64"], p, n, T, 11, 5, 0, hist=True)
    ib, bins = got["init_bins"], got["bins"]
    for i in range(p.n_initial):
        assert np.array_equal(got["hist_initial"][i], np.bincount(ib[:, i] - 1, minlength=64)), i
    for d in range(bins.shape[1]):
        assert np.array_equal(got["hist_transition"][d], np.bincount(bins[:, d, 1:].ravel() - 1, minlength=64)), d
    assert got["hist_initial"][0, 63] > 0 and got["hist_transition"][0, 63] > 0, "bin 64 never drawn"


def oracle_rows(samples):
    """the Python oracle's event lists back to back: dt, var, bin (int64), value (float64), offsets"""
    ev = [s.events for s in samples]
    off = np.concatenate(([0], np.cumsum([len(e) for e in ev]))).astype(np.int64)
    allev = np.concatenate(ev)
    bins = np.concatenate([s.event_bins for s in samples]).astype(np.int64)
    return allev[:, 0].astype(np.int64), allev[:, 1].astype(np.int64), bins, allev[:, 2], off


@pytest.mark.parametrize("name", EVENTS)
def test_emu_event_rows_equal_python_oracle(paths, name):
    """8-byte emb_event rows from the packed write pass (4-bit gated ordinals on deep_step) against the oracle's lists"""
    p = em_read(paths[name])
    n, T = 24, 40
    ev, off = H.EmuModel(paths[name]).sample_events(n, T, 13, FIRST, H.EmuModel.opts(p.n_initial))
    dt, var, bins, val, woff = oracle_rows(dbn_tracks(p, n, T, KeyedPhilox(13), first_sample=FIRST))
    assert np.array_equal(off, woff), "rows per track differ"
    assert np.array_equal(ev["dt"].astype(np.int64), dt) and np.array_equal(ev["var"].astype(np.int64), var)
    assert np.array_equal(ev["bin"].astype(np.int64), bins)
    assert np.all(np.abs(ev["value"].astype(np.float64) - val) <= 1e-6 * np.abs(val))


@pytest.mark.parametrize("name", ["wide_frozen", "hist64"])
def test_emu_event_rows_refused_above_16_bins(paths, name):
    p = em_read(paths[name])
    with pytest.raises(L.EmbError) as ei:
        H.EmuModel(paths[name]).sample_events(4, 8, 1, 0, H.EmuModel.opts(p.n_initial))
    assert ei.value.code == L.EMB_E_LIMIT


@pytest.mark.parametrize("correct_dbn", [False, True], ids=["sampler_branch", "correct_dbn"])
@pytest.mark.parametrize("name", DBN)
def test_emu_scores_equal_oracle(paths, name, correct_dbn):
    """emb_loglik_initial / _tracks / _track_events on oracle-sampled tracks against oracle/loglik*.py"""
    p = em_read(paths[name])
    n, T = 40, 25
    ref = COracle(p).sample_tracks(n, T, seed=17, first_sample=FIRST, threads=0)
    dyn, _ = layout(p)
    ib, bins = ref["init_bins"], ref["sample_bins"][:, dyn, :]
    em = TE.EmuModel(paths[name])
    gi, gt = TE.emu_dense(em, ib, bins, correct_dbn)
    wi, wt = OL.loglik_tracks(p, ib, bins, correct_dbn=correct_dbn)
    TE.assert_same(gi, wi)
    TE.assert_same(gt, wt)
    total, pv = TL.emu_initial(TL.EmuModel(paths[name]), ib)
    wtot, wpv = OL.loglik_initial(p, ib)
    assert np.array_equal(total, gi)
    TE.assert_same(pv, wpv)
    if name == "wide_frozen":
        return
    dt, var, ebins, _, off = oracle_rows(dbn_tracks(p, n, T, KeyedPhilox(17), first_sample=FIRST))
    ei, et = TE.emu_events(em, ib, dt, var, ebins, off, T, correct_dbn)
    wi, wt = OE.loglik_track_events(p, ib, dt, var, ebins, off, T, correct_dbn=correct_dbn)
    TE.assert_same(ei, wi)
    TE.assert_same(et, wt)
    assert np.array_equal(ei, gi)


def test_emu_scoring_flags_a_bad_bin_of_a_high_ordinal_variable(paths):
    """a bin above r in the row of the 12th (last) gated variable of deep_step"""
    p = em_read(paths["deep_step"])
    em = TE.EmuModel(paths["deep_step"])
    v = em.m.gated_vars[-1]
    ib = np.ones((1, p.n_initial), dtype=np.int8)
    dt, var, bins, off = TE.lists([[(2, v, int(p.r_initial[v - 1]) + 1), (3, 0, 0)]])
    TE.emu_events(em, ib, dt, var, bins, off, 5, status=TE.BAD_BIN)


def test_emu_expand_and_format_with_8_dynamic_columns(paths):
    """emb_track_events_expand with its default 8 control columns and emb_format_em_sample's 8-column transition.txt rows"""
    p = em_read(paths["deep_step"])
    n, T = 30, 40
    ev, off = H.EmuModel(paths["deep_step"]).sample_events(n, T, 19, FIRST, H.EmuModel.opts(p.n_initial))
    ref = COracle(p).sample_tracks(n, T, seed=19, first_sample=FIRST, threads=0)
    iv = ref["init_values"]
    em = TX.EmuModel(paths["deep_step"])
    assert em.m.n_dyn == 8
    smp, ctl = TX.emu_expand(em, iv, ev, None, off, T, packed=False)
    TX.check_against_host(em, iv, ev["dt"], ev["var"], ev["value"].astype(np.float64), off, T, smp, ctl)
    assert all(c.shape[1] == 9 for c in ctl)

    dyn, tv = layout(p)
    got, _ = emu_tracks(paths["deep_step"], p, n, T, 19, FIRST, 0)
    cols = [tv.index(d) for d in dyn]
    text, _ = emu_text(n, T, 7, p.n_initial, cols, len(tv), None, tile(np.asarray(got["values"], np.float32)), True)
    assert text == rows_transition(np.asarray(got["values"], np.float64)[:, cols, :], 7).encode()


# ---- the array constructor and the limits ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(LM.CASES))
def test_from_arrays_packs_the_file_model(paths, name):
    p = em_read(paths[name])
    kw = dict(boundaries=p.boundaries, resample_rates=p.resample_rates)
    if p.n_transition:
        kw.update(G_transition=p.G_transition, r_transition=p.r_transition, N_transition=p.N_transition,
                  temporal_map=p.temporal_map)
    a = EncounterModel.from_arrays(p.G_initial, p.r_initial, p.N_initial, **kw)
    f = EncounterModel(paths[name])
    for which in (0, 1):
        assert np.array_equal(a.packed(which), f.packed(which)), which
    assert a.gated_vars == f.gated_vars and a.order_transition == f.order_transition


def uniform_model(n, r=2, n_dyn=0, parents_of_last=0, rates=0.0):
    """n independent variables of r bins (the last with `parents_of_last` parents) and n_dyn dynamic copies"""
    G = np.zeros((n, n))
    G[:parents_of_last, n - 1] = 1
    N = [np.ones((r, 1))] * (n - 1) + [np.ones((r, r ** parents_of_last))]
    kw = dict(resample_rates=np.full(n, rates))
    if n_dyn:
        nt = n + n_dyn
        Gt = np.zeros((nt, nt))
        for k in range(n_dyn):
            Gt[k, n + k] = 1
        kw.update(G_transition=Gt, r_transition=[r] * nt, N_transition=[None] * n + [np.ones((r, r))] * n_dyn,
                  temporal_map=[[k + 1, n + k + 1] for k in range(n_dyn)])
    return EncounterModel.from_arrays(G, [r] * n, N, **kw)


def test_models_at_every_limit_load():
    m = uniform_model(L.EMB_MAX_VARS, r=127, n_dyn=L.EMB_MAX_DYN)
    assert (m.n_initial, m.n_dyn, max(m.r_initial)) == (L.EMB_MAX_VARS, L.EMB_MAX_DYN, 127)
    m = uniform_model(L.EMB_MAX_GATED, parents_of_last=L.EMB_MAX_PARENTS, rates=0.5)
    assert m.n_gated == L.EMB_MAX_GATED and int(m.G_initial.sum(axis=0).max()) == L.EMB_MAX_PARENTS


ONE_PAST = {
    "25 variables": (lambda: uniform_model(L.EMB_MAX_VARS + 1), "more than EMB_MAX_VARS initial variables"),
    "9 dynamic": (lambda: uniform_model(10, n_dyn=L.EMB_MAX_DYN + 1), "more than EMB_MAX_DYN dynamic variables"),
    "9 parents": (lambda: uniform_model(10, parents_of_last=L.EMB_MAX_PARENTS + 1), "more than EMB_MAX_PARENTS parents"),
    "17 gated": (lambda: uniform_model(L.EMB_MAX_GATED + 1, rates=0.5), "more than EMB_MAX_GATED"),
    "128 bins": (lambda: uniform_model(3, r=128), "r_initial out of range [1,127]"),
}


@pytest.mark.parametrize("case", sorted(ONE_PAST))
def test_one_past_a_limit_is_refused(case):
    make, message = ONE_PAST[case]
    with pytest.raises(L.EmbError) as ei:
        make()
    assert ei.value.code == L.EMB_E_LIMIT and message in ei.value.message, ei.value.message
