"""GPU suite for models at the compiled limits (`-m gpu`, on the B200): the cases of tests/limit_models.py at 10^5..10^6
track-seconds through every device entry point -- sampling (host and device buffers, default and forced-generic routes),
histograms, event rows, scoring, expansion and formatting -- against the C oracle, the Python oracles and the host emulation.
Each case asserts the branch it reaches (test_model_limits.assert_branch, and the kernel the library reports it ran)."""
import numpy as np
import pytest

import limit_models as LM
import test_loglik as TL
import test_loglik_events as TE
from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel, controls_of, expand_events, untile_bins, untile_values
from oracle import loglik as OL
from oracle import loglik_events as OE
from oracle.c_oracle import COracle
from oracle.drivers import dbn_tracks
from oracle.em_read import em_read
from oracle.uniforms import KeyedPhilox
from test_format import rows_transition
from test_model_limits import DBN, EVENTS, TWINS, assert_branch, check_tracks, layout, oracle_rows, paths  # noqa: F401 (fixture)

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

FIRST = 2 ** 32 - 1000                    # every batch straddles sample 2^32
SIZE = {"wide_frozen": (3000, 60), "deep_step": (4000, 100), "hist64": (5000, 100), "fast_shape_twin": (6000, 120),
        "fast_shape_twin_step": (6000, 120)}


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _dense(m, res):
    """a TrackResult as the dict test_model_limits.check_tracks reads"""
    nd, ntv = len(res.dyn_vars), len(res.tv_vars)
    return dict(bins=untile_bins(_np(res.bins_tiled), nd, res.n, res.T), values=untile_values(_np(res.values_tiled), ntv, res.n, res.T),
                init_bins=_np(res.init_bins).T, init_values=_np(res.init_values).T, attempts=_np(res.attempts))


def _with_generic(fn):
    lib = L.lib()
    lib.emb_debug_force_generic(1)
    try:
        return fn()
    finally:
        lib.emb_debug_force_generic(0)


@pytest.fixture(scope="module")
def sampled(paths):
    """{name: (model, oracle parms, C-oracle result, device TrackResult)} for the cases with a transition network"""
    out = {}
    for name in DBN:
        m, p = EncounterModel(paths[name]), em_read(paths[name])
        n, T = SIZE[name]
        ref = COracle(p).sample_tracks(n, T, seed=31, first_sample=FIRST, threads=0)
        assert ref["rc"] == 0
        out[name] = (m, p, ref, m.sample_tracks(n, T, seed=31, first_sample=FIRST, device="cuda"))
    return out


@pytest.mark.parametrize("name", DBN)
def test_tracks_equal_c_oracle(paths, sampled, name):
    m, p, ref, res = sampled[name]
    assert_branch(name, m)
    n, T = SIZE[name]
    m.sample_tracks(n, T, seed=31, first_sample=FIRST, device="cuda")
    assert L.lib().emb_debug_last_kernel_fast() == (name in TWINS), "kernel route"
    check_tracks(_dense(m, res), ref, p)
    host = m.sample_tracks(n, T, seed=31, first_sample=FIRST)
    check_tracks(_dense(m, host), ref, p)
    generic = _with_generic(lambda: m.sample_tracks(n, T, seed=31, first_sample=FIRST, device="cuda"))
    assert L.lib().emb_debug_last_kernel_fast() == 0
    check_tracks(_dense(m, generic), ref, p)
    assert torch.equal(generic.bins_tiled, res.bins_tiled)


@pytest.mark.parametrize("name", sorted(LM.CASES))
def test_initial_equals_c_oracle(paths, name):
    """fp64 values bit for bit, fp32 values within 1e-6; the staging cases at n >= 2 * 148 * 1024"""
    m, p = EncounterModel(paths[name]), em_read(paths[name])
    assert_branch(name, m)
    n = 2 * 148 * 1024 + 5 if name.startswith("staging") else 100_003
    ref = COracle(p).sample_initial(n, seed=37, first_sample=FIRST, threads=0)
    assert ref["rc"] == 0
    fast = name in ("init15_wide", "staging_under", "staging_over", "fast_shape_twin", "fast_shape_twin_step")
    for device in ("cuda", None):
        bins, vals, att = m.sample_initial(n, seed=37, first_sample=FIRST, device=device)
        assert L.lib().emb_debug_last_kernel_fast() == fast
        assert np.array_equal(_np(bins), ref["bins"]) and np.array_equal(_np(vals), ref["values"])
        assert np.all(_np(att) == 1)
    bins, v32, _ = m.sample_initial(n, seed=37, first_sample=FIRST, device="cuda", values_fp32=True)
    assert np.array_equal(_np(bins), ref["bins"])
    w = ref["values"]
    assert np.all(np.abs(_np(v32).astype(np.float64) - w) <= 1e-6 * np.abs(w))
    if name != "init15_wide":
        bins, vals, _ = _with_generic(lambda: m.sample_initial(n, seed=37, first_sample=FIRST, device="cuda"))
        assert L.lib().emb_debug_last_kernel_fast() == 0
        assert np.array_equal(_np(bins), ref["bins"]) and np.array_equal(_np(vals), ref["values"])
    # scoring of the same states: k_loglik_initial (staged or gathered table) against the emulation and the oracle
    total, pv = m.loglik_initial(bins, per_var=True)
    wt, wpv = TL.emu_initial(TL.EmuModel(paths[name]), _np(bins))
    assert np.array_equal(_np(total), wt) and np.array_equal(_np(pv), wpv)
    TE.assert_same(_np(total), OL.loglik_initial(p, _np(bins))[0])


def test_histograms_at_the_stride(paths, sampled):
    m, p, ref, _ = sampled["hist64"]
    n, T = SIZE["hist64"]
    hi = torch.zeros((m.n_initial, 64), dtype=torch.int64, device="cuda")
    ht = torch.zeros((m.n_dyn, 64), dtype=torch.int64, device="cuda")
    m.sample_tracks(n, T, seed=31, first_sample=FIRST, device="cuda", hist_initial=hi, hist_transition=ht)
    dyn, _ = layout(p)
    for i in range(p.n_initial):
        assert np.array_equal(_np(hi[i]), np.bincount(ref["init_bins"][:, i] - 1, minlength=64)), i
    for d, v in enumerate(dyn):
        assert np.array_equal(_np(ht[d]), np.bincount(ref["sample_bins"][:, v, 1:].ravel() - 1, minlength=64)), d
    assert int(hi[0, 63]) > 0 and int(ht[0, 63]) > 0


@pytest.mark.parametrize("name", DBN)
def test_event_rows(paths, sampled, name):
    m, p, ref, _ = sampled[name]
    n, T = SIZE[name]
    if name not in EVENTS:
        with pytest.raises(L.EmbError) as ei:
            m.sample_events(n, T, seed=31, first_sample=FIRST, device="cuda")
        assert ei.value.code == L.EMB_E_LIMIT
        return
    k = 150                                                 # tracks checked row by row against the Python oracle
    dt, var, bins, val, woff = oracle_rows(dbn_tracks(p, k, T, KeyedPhilox(31), first_sample=FIRST))
    for device in ("cuda", None):
        ev = m.sample_events(n, T, seed=31, first_sample=FIRST, device=device)
        off = _np(ev.offsets)
        rows = _np(ev.events).view(L.EVENT_DTYPE).reshape(-1)
        assert np.array_equal(np.diff(off), ref["n_events"]) and off[0] == 0 and off[-1] == ev.total
        a = rows[:woff[-1]]
        assert np.array_equal(off[:k + 1], woff)
        assert np.array_equal(a["dt"].astype(np.int64), dt) and np.array_equal(a["var"].astype(np.int64), var)
        assert np.array_equal(a["bin"].astype(np.int64), bins)
        assert np.all(np.abs(a["value"].astype(np.float64) - val) <= 1e-6 * np.abs(val))
        assert np.array_equal(_np(ev.init_bins).T, ref["init_bins"])
    if m.n_gated > 7:
        with pytest.raises(L.EmbError) as ei:
            m.sample_events_packed(n, T, seed=31, first_sample=FIRST, device="cuda")
        assert ei.value.code == L.EMB_E_LIMIT
        return
    pk = m.sample_events_packed(n, T, seed=31, first_sample=FIRST, device="cuda")
    assert np.array_equal(_np(pk.offsets), off)
    pdt, pvar, pbin, pval = pk.decode()
    assert np.array_equal(pdt[:woff[-1]], dt) and np.array_equal(pvar[:woff[-1]], var) and np.array_equal(pbin[:woff[-1]], bins)
    assert np.all(np.abs(pval[:woff[-1]] - val) <= 1e-12 * np.abs(val))


@pytest.mark.parametrize("correct_dbn", [False, True], ids=["sampler_branch", "correct_dbn"])
@pytest.mark.parametrize("name", DBN)
def test_scores(paths, sampled, name, correct_dbn):
    m, p, ref, res = sampled[name]
    n, T = SIZE[name]
    di, dtr = m.loglik_tracks(res, correct_dbn=correct_dbn)
    dyn, _ = layout(p)
    ib, bins = ref["init_bins"], ref["sample_bins"][:, dyn, :]
    em = TE.EmuModel(paths[name])
    wi, wt = TE.emu_dense(em, ib, bins, correct_dbn)
    assert np.array_equal(_np(di), wi) and np.array_equal(_np(dtr), wt), "device != host emulation"
    oi, ot = OL.loglik_tracks(p, ib, bins, correct_dbn=correct_dbn)
    TE.assert_same(_np(di), oi)
    TE.assert_same(_np(dtr), ot)
    if name not in EVENTS:
        return
    ev = m.sample_events(n, T, seed=31, first_sample=FIRST, device="cuda")
    ei, et = m.loglik_events(ev, correct_dbn=correct_dbn)
    rows = _np(ev.events).view(L.EVENT_DTYPE).reshape(-1)
    off = _np(ev.offsets)
    gi, gt = TE.emu_events(em, ib, rows["dt"], rows["var"], rows["bin"], off, T, correct_dbn)
    assert np.array_equal(_np(ei), gi) and np.array_equal(_np(et), gt), "event scoring: device != host emulation"
    k = 300
    oi, ot = OE.loglik_track_events(p, ib[:k], rows["dt"], rows["var"], rows["bin"], off[:k + 1], T, correct_dbn=correct_dbn)
    TE.assert_same(_np(ei)[:k], oi)
    TE.assert_same(_np(et)[:k], ot)
    if name == "deep_step" and not correct_dbn:
        v = m.gated_vars[-1]                                # the 12th gated variable (a 4-bit ordinal in the write pass)
        bad = rows.copy()
        j = int(np.nonzero(bad["var"] == v)[0][0])
        bad["bin"][j] = int(m.r_initial[v - 1]) + 1
        with pytest.raises(L.EmbError) as exc:
            m.loglik_events(torch.from_numpy(bad.view(np.int64)).cuda(), ev.offsets, T, ev.init_bins)
        assert exc.value.code == L.EMB_E_ARG and "outside 1..r" in exc.value.message


def test_expand_and_format_with_8_dynamic_columns(sampled):
    m, p, ref, res = sampled["deep_step"]
    n, T = SIZE["deep_step"]
    ev = m.sample_events(n, T, seed=31, first_sample=FIRST, device="cuda")
    smp, ctl = m.expand_events_gpu(ev)
    rows = _np(ev.events).view(L.EVENT_DTYPE).reshape(-1)
    off = _np(ev.offsets)
    iv = _np(ev.init_values).T
    dense = expand_events(iv, rows["dt"], rows["var"], rows["value"].astype(np.float64), off, T)
    assert np.array_equal(_np(smp), dense.transpose(0, 2, 1))
    want = controls_of(dense, rows["dt"], off, np.asarray(m.temporal_map)[:, 0] - 1)
    got_rows, got_off = _np(ctl.rows), _np(ctl.offsets)
    assert got_rows.shape[1] == 9 and np.array_equal(np.diff(got_off), [len(w) for w in want])
    assert np.array_equal(got_rows, np.concatenate(want))

    k = 400
    small = m.sample_tracks(k, T, seed=31, first_sample=FIRST, device="cuda")
    _, _, text, toff = m.format_em_sample(small, first_id=2 ** 40)
    dyn, tv = layout(p)
    vals = _dense(m, small)["values"].astype(np.float64)[:, [tv.index(d) for d in dyn], :]
    assert _np(text).tobytes() == rows_transition(vals, 2 ** 40).encode()
    assert int(_np(toff)[-1]) == len(_np(text))
