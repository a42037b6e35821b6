"""CPU suite: the device sampling routines (emb_device.cuh), executed on the host by the TEST-ONLY
emulation in tests/emu, against the oracle's golden vectors.  The GPU suite (test_gpu_parity.py) runs
the same cases through libemb200.so on a B200."""
import numpy as np
import pytest

import cases
from em_model_manned_bayes_b200 import _lib as L
import helpers as H
from helpers import EmuModel
from oracle.em_read import em_read


def _model_and_opts(model_paths, c):
    path = model_paths[c["model"]]
    ow = c.get("overwrite", ())
    p = em_read(path, isOverwriteZeroBoundaries=bool(ow), idxZeroBoundaries=ow or (1, 2, 3))
    em = EmuModel(path, idx_zero=ow, overwrite=bool(ow))
    if c.get("prior") == "dbe":
        em.set_prior(0, L.EMB_PRIOR_DBE, 0.0)
        em.set_prior(1, L.EMB_PRIOR_DBE, 0.0)
    kw = {}
    if c["uncor"]:
        lab = p.labels_initial
        kw.update(reject_mode=L.EMB_REJECT_UNCOR, idx_v=cases.label_index(lab, '"v"'),
                  idx_dh=cases.label_index(lab, '"\\dot h"'), idx_L=cases.label_index(lab, '"L"'))
        if c.get("q500"):
            kw["is_quantize500"] = 1
        if c.get("layers") is not None:
            kw["layers"] = c["layers"]
    return p, em, EmuModel.opts(p.n_initial, start=c.get("start"), **kw)


def _run_tracks(model_paths, c):
    p, em, o = _model_and_opts(model_paths, c)
    nd = p.temporal_map.shape[0]
    ntv = len(set(p.temporal_map[:, 0]) | {i + 1 for i in range(p.n_initial) if p.resample_rates[i] > 0})
    return em.sample_tracks(p.n_initial, nd, ntv, c["n"], c["T"], c["seed"], c.get("first", 0), o)


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "specialised"])
@pytest.mark.parametrize("name", sorted(cases.TRACK_CASES))
def test_tracks_match_golden(model_paths, golden, name, fast):
    """Both device code paths (track_generic and the register-resident track_fast) against the oracle."""
    from helpers import emu_lib
    lib = emu_lib()
    lib.emu_use_fast(fast)
    try:
        got = _run_tracks(model_paths, cases.TRACK_CASES[name])
        used_fast = lib.emu_last_fast()
    finally:
        lib.emu_use_fast(0)
    cases.check_tracks(got, golden[name])
    assert used_fast == fast, "every golden model shape is expected to have a specialised kernel"


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "specialised"])
@pytest.mark.parametrize("name", sorted(cases.TRACK_CASES))
def test_event_lists_match_golden(model_paths, golden, name, fast):
    """out_events (dbn_hierarchical_sample.m:9-37): rows, order, dt, variable and bin identical to the oracle."""
    from helpers import emu_lib
    lib = emu_lib()
    c = cases.TRACK_CASES[name]
    p, em, o = _model_and_opts(model_paths, c)
    lib.emu_use_fast(fast)
    try:
        ev, off = em.sample_events(c["n"], c["T"], c["seed"], c.get("first", 0), o)
        assert lib.emu_last_fast() == fast
    finally:
        lib.emu_use_fast(0)
    cases.check_events(ev, off, golden[name])


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "specialised"])
@pytest.mark.parametrize("name", sorted(cases.INITIAL_CASES))
def test_initial_matches_golden(model_paths, golden, name, fast):
    from helpers import emu_lib
    lib = emu_lib()
    c = cases.INITIAL_CASES[name]
    p = em_read(model_paths[c["model"]])
    em = EmuModel(model_paths[c["model"]])
    lib.emu_use_fast(fast)
    try:
        bins, vals, att = em.sample_initial(p.n_initial, c["n"], c["seed"], c["first"], EmuModel.opts(p.n_initial))
        assert lib.emu_last_fast() == fast
    finally:
        lib.emu_use_fast(0)
    assert np.array_equal(bins, golden[name]["bins"])
    assert np.array_equal(vals, golden[name]["values"])
    assert np.all(att == 1)


@pytest.mark.parametrize("model,n,start", [
    ("balloon_v1", 37, None), ("glider_v1", 1001, None), ("glider_v1", 64, [2, None, None, None, None]),
    ("littoral_uncor_v1", 130, None), ("uncor_1200code_v2p1", 203, [1, 4, 2, None, None, None, None]),
    ("terminal_v3_radar_encounter_model", 95, None), ("cor_v1", 50, None)])
@pytest.mark.parametrize("first", [5, 8, 2 ** 34 - 6], ids=["unaligned", "aligned", "group-high-word-changes"])
def test_initial_specialised_equals_generic(model_paths, model, n, start, first):
    """initial_fast4 (4 samples per thread, register state) == sample_initial, ragged n and presets included;
    cor_v1 has a non-identity topological order and must fall back to the generic routine.  Stream spec v5 lets four
    consecutive samples share their Philox calls: first_sample not a multiple of four (two calls per variable) and a
    batch whose sample >> 2 crosses a multiple of 2^32 (the shared call table no longer applies) are the edge cases."""
    from helpers import emu_lib
    lib = emu_lib()
    p = em_read(model_paths[model])
    em = EmuModel(model_paths[model])
    o = EmuModel.opts(p.n_initial, start=start)
    ref = em.sample_initial(p.n_initial, n, 21, first, o)
    lib.emu_use_fast(1)
    try:
        got = em.sample_initial(p.n_initial, n, 21, first, o)
        assert lib.emu_last_fast() == (0 if model == "cor_v1" else 1)
    finally:
        lib.emu_use_fast(0)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name", sorted(cases.TERMINAL_CASES))
def test_terminal_geometry_matches_golden(model_paths, golden, name):
    c = cases.TERMINAL_CASES[name]
    p = em_read(model_paths[c["model"]])
    em = EmuModel(model_paths[c["model"]])
    lo, hi = [-np.inf] * p.n_initial, [np.inf] * p.n_initial
    for lab in ('"own_speed"', '"int_speed"'):
        i = p.labels_initial.index(lab)
        lo[i], hi[i] = cases.GENERIC_VEL
    o = EmuModel.opts(p.n_initial, start=c["start"], reject_mode=L.EMB_REJECT_BOX, box_lo=lo, box_hi=hi)
    bins, vals, att = em.sample_initial(p.n_initial, c["n"], c["seed"], 0, o)
    assert np.array_equal(bins, golden[name]["bins"])
    assert np.array_equal(vals, golden[name]["values"])
    assert np.array_equal(att.astype(np.int64), golden[name]["attempts"].astype(np.int64))


def test_shard_invariance(model_paths):
    """Results are keyed by the global sample index: [0,40) == [0,13) + [13,40)."""
    c = dict(cases.TRACK_CASES["uncor_v2p1_n24_T300_seed1"], n=40, T=64)
    whole = _run_tracks(model_paths, c)
    a = _run_tracks(model_paths, dict(c, n=13))
    b = _run_tracks(model_paths, dict(c, n=27, first=13))
    for k in ("bins", "values", "init_bins", "init_values"):
        assert np.array_equal(np.concatenate([a[k], b[k]]), whole[k]), k


def test_histograms_count_every_column(model_paths):
    path = model_paths["uncor_1200code_v2p1"]
    p = em_read(path)
    em = EmuModel(path)
    o = EmuModel.opts(p.n_initial)
    r = em.sample_tracks(p.n_initial, 3, 4, 50, 37, 9, 0, o, hist=True)
    assert r["hist_initial"].sum(axis=1).tolist() == [50] * 7
    assert r["hist_transition"].sum(axis=1).tolist() == [50 * 36] * 3
    for d in range(3):
        cnt = np.bincount(r["bins"][:, d, 1:].ravel() - 1, minlength=64)
        assert np.array_equal(cnt, r["hist_transition"][d])


def test_preset_dependent_variable_is_rejected(model_paths):
    p = em_read(model_paths["uncor_1200code_v2p1"])
    em = EmuModel(model_paths["uncor_1200code_v2p1"])
    o = EmuModel.opts(p.n_initial, start=[None, 2, None, None, None, None, None])
    with pytest.raises(L.EmbError, match="Attempt to preset a dependent variable"):
        em.sample_initial(p.n_initial, 4, 1, 0, o)


@pytest.mark.parametrize("model,uncor,n,T", [("uncor_allcode_fwsingle_v1", True, 300, 600), ("glider_v1", True, 400, 150),
                                             ("cor_v1", False, 300, 60), ("uncor_1200only_fwse_v1p2", True, 300, 100),
                                             ("fai1_v1", True, 300, 100), ("uncor_1200code_v1", True, 200, 100),
                                             ("blimp_v1", True, 300, 100), ("dueregard_v1", True, 200, 100),
                                             ("haa_v1", True, 200, 100), ("littoral_cor_v1", False, 200, 60),
                                             ("weatherballoon_v1", False, 300, 60)])
@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "specialised"])
def test_tracks_match_c_oracle(model_paths, model, uncor, n, T, fast):
    """Host emulation of the device code against the plain-C restatement at a few 10^4..10^5 track-seconds."""
    from oracle.c_oracle import COracle
    from oracle.em_read import em_read
    p = em_read(model_paths[model])
    ref = COracle(p, uncor=uncor).sample_tracks(n, T, seed=92, first_sample=7 * 10 ** 10, threads=0)
    assert ref["rc"] == 0
    lib = H.emu_lib()
    lib.emu_use_fast(fast)
    m = H.EmuModel(model_paths[model])
    kw = {}
    if uncor:
        lab = p.labels_initial
        kw = dict(reject_mode=L.EMB_REJECT_UNCOR, idx_v=cases.label_index(lab, '"v"'), idx_dh=cases.label_index(lab, '"\\dot h"'),
                  idx_L=cases.label_index(lab, '"L"'))
    tm = np.asarray(p.temporal_map)
    dyn = [int(v) - 1 for v in tm[:, 0]]
    rates = np.asarray(p.resample_rates)
    tv = sorted(set(dyn) | {i for i in range(p.n_initial) if rates[i] > 0})
    got = m.sample_tracks(p.n_initial, len(dyn), len(tv), n, T, 92, 7 * 10 ** 10, H.EmuModel.opts(p.n_initial, **kw))
    assert lib.emu_last_fast() == fast, "every shipped model shape has a specialised kernel (EMB_FAST_SHAPES)"
    lib.emu_use_fast(0)
    assert np.array_equal(got["init_bins"], ref["init_bins"]) and np.array_equal(got["init_values"], ref["init_values"])
    assert np.array_equal(got["attempts"].astype(np.int64), ref["attempts"].astype(np.int64))
    assert np.array_equal(got["bins"], ref["sample_bins"][:, dyn, :])
    want = ref["samples"][:, tv, :]
    assert np.all(np.abs(got["values"].astype(np.float64) - want) <= 1e-6 * np.abs(want))


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "specialised"])
def test_tracks_across_a_2_32_sample_boundary(model_paths, fast):
    """Stream spec v4 puts sample >> 32 into counter word 0, which the specialised kernel treats as launch-uniform
    (philox_track / philox_call): a call whose global sample indices straddle a multiple of 2^32 is split into two
    launches (next_segment).  Tracks on both sides of the boundary must match the C restatement."""
    from oracle.c_oracle import COracle
    from oracle.em_read import em_read
    p = em_read(model_paths["uncor_1200code_v2p1"])
    n, T, first = 90, 40, 3 * 2 ** 32 - 37
    ref = COracle(p, uncor=True).sample_tracks(n, T, seed=5, first_sample=first, threads=0)
    lib = H.emu_lib()
    lib.emu_use_fast(fast)
    m = H.EmuModel(model_paths["uncor_1200code_v2p1"])
    lab = p.labels_initial
    kw = dict(reject_mode=L.EMB_REJECT_UNCOR, idx_v=cases.label_index(lab, '"v"'), idx_dh=cases.label_index(lab, '"\\dot h"'),
              idx_L=cases.label_index(lab, '"L"'))
    tm = np.asarray(p.temporal_map)
    dyn = [int(v) - 1 for v in tm[:, 0]]
    rates = np.asarray(p.resample_rates)
    tv = sorted(set(dyn) | {i for i in range(p.n_initial) if rates[i] > 0})
    got = m.sample_tracks(p.n_initial, len(dyn), len(tv), n, T, 5, first, H.EmuModel.opts(p.n_initial, **kw))
    assert lib.emu_last_fast() == fast
    lib.emu_use_fast(0)
    assert np.array_equal(got["init_bins"], ref["init_bins"])
    assert np.array_equal(got["bins"], ref["sample_bins"][:, dyn, :])
    want = ref["samples"][:, tv, :]
    assert np.all(np.abs(got["values"].astype(np.float64) - want) <= 1e-6 * np.abs(want))


@pytest.mark.skipif(not H.have_reference(), reason="needs EMB200_REFERENCE_DIR (an upstream checkout with model/*.txt)")
def test_every_shipped_dbn_model_runs_specialised_and_matches_the_c_oracle():
    """All model/*.txt files with a transition network (not just the archived ones): the specialised code path
    (EMB_FAST_SHAPES covers every shipped shape and sampling order) against the plain-C restatement."""
    import glob
    import os
    from oracle.c_oracle import COracle
    lib = H.emu_lib()
    seen = 0
    for path in sorted(glob.glob(os.path.join(H.REF_MODEL_DIR, "*.txt"))):
        p = em_read(path)
        if not p.n_transition:
            continue
        n, T = 60, 80
        ref = COracle(p).sample_tracks(n, T, seed=93, first_sample=3 * 10 ** 9, threads=0)
        assert ref["rc"] == 0
        tm = np.asarray(p.temporal_map)
        dyn = [int(v) - 1 for v in tm[:, 0]]
        rates = np.asarray(p.resample_rates)
        tv = sorted(set(dyn) | {i for i in range(p.n_initial) if rates[i] > 0})
        lib.emu_use_fast(1)
        try:
            got = H.EmuModel(path).sample_tracks(p.n_initial, len(dyn), len(tv), n, T, 93, 3 * 10 ** 9, H.EmuModel.opts(p.n_initial))
            assert lib.emu_last_fast() == 1, "no specialised kernel for " + os.path.basename(path)
        finally:
            lib.emu_use_fast(0)
        assert np.array_equal(got["init_bins"], ref["init_bins"]), path
        assert np.array_equal(got["bins"], ref["sample_bins"][:, dyn, :]), path
        want = ref["samples"][:, tv, :]
        assert np.all(np.abs(got["values"].astype(np.float64) - want) <= 1e-6 * np.abs(want)), path
        seen += 1
    assert seen >= 20


@pytest.mark.parametrize("fast", [0, 1], ids=["generic", "specialised"])
def test_correct_dbn_option_matches_the_oracle(model_paths, fast):
    """emb_sample_opts::correct_dbn (SURVEY 8f row 2; NOT the reference's default): for a model without a dynamic -> dynamic
    edge the parents of the dynamic variables are re-evaluated every second (dbn_sample.m:66-79) instead of frozen at t = 1
    (:110-135).  Against the oracle with the same option; and the option really changes the tracks."""
    from oracle.drivers import uncor_sample
    from oracle.uniforms import KeyedPhilox
    p = em_read(model_paths["uncor_1200code_v2p1"])
    n, T = 40, 120
    want = uncor_sample(p, n, T, KeyedPhilox(6), correct_dbn=True)
    bins, vals, dyn, tv = H.oracle_dense(p, want)
    frozen = H.oracle_dense(p, uncor_sample(p, n, T, KeyedPhilox(6)))[0]
    assert not np.array_equal(bins, frozen)
    lib = H.emu_lib()
    lib.emu_use_fast(fast)
    m = H.EmuModel(model_paths["uncor_1200code_v2p1"])
    lab = p.labels_initial
    o = H.EmuModel.opts(p.n_initial, reject_mode=L.EMB_REJECT_UNCOR, idx_v=cases.label_index(lab, '"v"'),
                        idx_dh=cases.label_index(lab, '"\\dot h"'), idx_L=cases.label_index(lab, '"L"'), correct_dbn=1)
    got = m.sample_tracks(p.n_initial, 3, 4, n, T, 6, 0, o)
    assert lib.emu_last_fast() == fast
    lib.emu_use_fast(0)
    assert np.array_equal(got["bins"], bins)
    assert np.all(np.abs(got["values"].astype(np.float64) - vals) <= 1e-6 * np.abs(vals))
