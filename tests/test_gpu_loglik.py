"""GPU suite for the log-likelihood entry points (`-m gpu`, on the B200): k_loglik_initial / k_loglik_tracks against the host
emulation of the same code bit for bit, host against device buffers, the status-word errors, and two statistical identities
that check the whole joint law the samplers draw from: the mean log-likelihood of sampled states and tracks against the exact
(negative) entropies from enumerating the initial network, and self-normalised importance sampling from a flattened
proposal reproducing the exact marginals."""
import itertools

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel
from oracle import loglik as OL
from oracle.em_read import em_read
from test_loglik import EmuModel, assert_same, emu_initial, emu_tracks

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

UNCOR = "uncor_allcode_fwsingle_v1"


def _sample(m, n, T, seed, **kw):
    res = m.sample_tracks(n, T, seed=seed, device="cuda", want_values=False, **kw)
    return res


def _device_vs_emu(model_paths, model, n, T, seed, correct_dbn=False):
    m = EncounterModel(model_paths[model])
    res = _sample(m, n, T, seed)
    init, trans = m.loglik_tracks(res, correct_dbn=correct_dbn)
    em = EmuModel(model_paths[model])
    ib = res.init_bins.cpu().numpy().T
    bins = res.bins.cpu().numpy()
    wi, wt = emu_tracks(em, ib, bins, correct_dbn=correct_dbn)
    gi, gt = init.cpu().numpy(), trans.cpu().numpy()
    assert np.array_equal(gi, wi), "initial term: device != host emulation"
    assert np.array_equal(gt, wt), "transition term: device != host emulation"
    return m, res, gi, gt


def test_fast_branch_matches_emulation(model_paths):
    """20 000 x 600 s of the flagship model: the counting kernel (frozen parents) bit for bit"""
    m, _, gi, gt = _device_vs_emu(model_paths, UNCOR, 20_000, 600, seed=101)
    assert not m.is_dynvar_depend
    assert np.isfinite(gi).all() and np.isfinite(gt).all()


@pytest.mark.parametrize("model,n,T", [("glider_v1", 5_000, 120), ("cor_v1", 3_000, 60), ("balloon_v1", 4_000, 50)])
def test_other_models_match_emulation(model_paths, model, n, T):
    _device_vs_emu(model_paths, model, n, T, seed=202)


@pytest.mark.parametrize("model", [UNCOR, "glider_v1"])
def test_correct_dbn_matches_emulation(model_paths, model):
    _device_vs_emu(model_paths, model, 3_000, 99, seed=303, correct_dbn=True)


def test_glider_initial_matches_emulation(model_paths):
    """100 000 samples: enough for the shared-memory staged table"""
    m = EncounterModel(model_paths["glider_v1"])
    bins, _, _ = m.sample_initial(100_000, seed=404, device="cuda", want_values=False, want_attempts=False)
    total, pv = m.loglik_initial(bins, per_var=True)
    wt, wpv = emu_initial(EmuModel(model_paths["glider_v1"]), bins.cpu().numpy())
    assert np.array_equal(total.cpu().numpy(), wt)
    assert np.array_equal(pv.cpu().numpy(), wpv)
    assert_same(total.cpu().numpy(), OL.loglik_initial(em_read(model_paths["glider_v1"]), bins.cpu().numpy())[0])


def test_host_buffers_equal_device_buffers(model_paths):
    m = EncounterModel(model_paths["cor_v1"])
    res = _sample(m, 1_000, 37, seed=505)
    di, dt = m.loglik_tracks(res)
    hi, ht = m.loglik_tracks(res.init_bins.cpu().numpy(), res.bins_tiled.cpu().numpy(), 37)
    assert isinstance(hi, np.ndarray) and np.array_equal(hi, di.cpu().numpy()) and np.array_equal(ht, dt.cpu().numpy())
    b = res.init_bins.T
    assert np.array_equal(m.loglik_initial(b.cpu().numpy()), m.loglik_initial(b).cpu().numpy())


def test_device_status_word_reports_bad_input(model_paths):
    m = EncounterModel(model_paths["glider_v1"])
    res = _sample(m, 300, 10, seed=606)
    bad = res.bins_tiled.clone()
    bad[bad == 2] = 77                                       # out of range somewhere past column 0
    with pytest.raises(L.EmbError) as ei:
        m.loglik_tracks(res.init_bins, bad, 10)
    assert ei.value.code == L.EMB_E_ARG and "outside 1..r" in ei.value.message
    ib = res.init_bins.clone()
    d0 = int(m.temporal_map[0, 0]) - 1
    ib[d0] = torch.where(ib[d0] == 1, 2, 1).to(torch.int8)  # column 0 no longer equals the initial state
    with pytest.raises(L.EmbError) as ei:
        m.loglik_tracks(ib, res.bins_tiled, 10)
    assert ei.value.code == L.EMB_E_ARG and "column 0" in ei.value.message


# ---- exact expectations from enumerating the initial network ----------------------------------------------------------
def _enumerate(p):
    """all joint configurations (rows, 1-based) of the initial network and log p of each"""
    X = np.array(list(itertools.product(*[range(1, int(r) + 1) for r in p.r_initial])), dtype=np.int64)
    lp, per = OL.loglik_initial(p, X)
    return X, lp, per


def test_mean_loglik_matches_exact_entropy(model_paths):
    """1.25M x 600 s tracks of the flagship model (no rejection): mean initial term == -H(X) and mean transition term ==
    -(T-1) E[sum_k H(X_k | pa_0)], within 5 standard errors estimated from the per-track spread"""
    p = em_read(model_paths[UNCOR])
    X, lp, _ = _enumerate(p)
    assert X.shape[0] == 125_440
    px = np.exp(lp)
    assert abs(px.sum() - 1.0) < 1e-9
    with np.errstate(invalid="ignore"):                      # 0 * -inf in the configurations of probability 0
        neg_H = float(np.sum(np.where(px > 0, px * lp, 0.0)))
    # per configuration: sum over the dynamic variables of sum_b P log P in the frozen column
    tm = np.asarray(p.temporal_map)
    X0 = np.ones((X.shape[0], p.n_transition), dtype=np.int64)
    X0[:, :p.n_initial] = X
    for d in range(tm.shape[0]):
        X0[:, tm[d, 1] - 1] = X[:, tm[d, 0] - 1]
    e_step = np.zeros(X.shape[0])
    for d in range(tm.shape[0]):
        tab = OL.logp_table(p.N_transition[tm[d, 1] - 1])
        col = OL.parent_column(p.G_transition, p.r_transition, tm[d, 1] - 1, X0)
        P = np.exp(tab[:, col])
        with np.errstate(invalid="ignore"):
            e_step += np.sum(np.where(P > 0, P * tab[:, col], 0.0), axis=0)
    T = 600
    want_trans = (T - 1) * float(np.sum(px * e_step))

    m = EncounterModel(model_paths[UNCOR])
    n = 1_250_000
    res = _sample(m, n, T, seed=707)
    init, trans = m.loglik_tracks(res)
    assert torch.isfinite(init).all() and torch.isfinite(trans).all()
    for got, want in ((init, neg_H), (trans, want_trans)):
        mean, se = got.mean().item(), got.std().item() / np.sqrt(n)
        assert abs(mean - want) <= 5 * se, (mean, want, se)


def test_importance_sampling_reproduces_exact_marginals(model_paths):
    """10M initial states from a flattened proposal q (constant prior 1000), scored under p and q: self-normalised weights
    p/q reproduce p's exact marginals within 5 standard errors"""
    path = model_paths[UNCOR]
    p = em_read(path)
    X, lp, _ = _enumerate(p)
    px = np.exp(lp)
    mp = EncounterModel(path)
    mq = EncounterModel(path, prior=1000)
    n = 10_000_000
    bins, _, _ = mq.sample_initial(n, seed=808, device="cuda", want_values=False, want_attempts=False)
    lw = mp.loglik_initial(bins) - mq.loglik_initial(bins)
    w = torch.exp(lw - lw.max())
    W = w.sum()
    for i in range(p.n_initial):
        for b in range(1, int(p.r_initial[i]) + 1):
            exact = float(px[X[:, i] == b].sum())
            ind = (bins[:, i] == b).double()
            est = float((w * ind).sum() / W)
            se = float(torch.sqrt(((w * (ind - est)) ** 2).sum()) / W)
            assert abs(est - exact) <= 5 * se + 1e-12, (i, b, est, exact, se)
