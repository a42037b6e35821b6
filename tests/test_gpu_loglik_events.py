"""GPU suite for scoring tracks given as event lists (`-m gpu`, on the B200): k_loglik_events on the rows of sample_events and
sample_events_packed against the host emulation of the same code bit for bit, and against the dense scoring (emb_loglik_tracks)
of the same tracks from sample_tracks with the same seed; host against device buffers; the status-word refusals on corrupted
copies of real rows."""
import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel
from test_loglik_events import EmuModel, assert_same, emu_events

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

UNCOR = "uncor_allcode_fwsingle_v1"


def _host_rows(ev):
    return ev.events.cpu().numpy().view(L.EVENT_DTYPE)


def _check(model_paths, model, n, T, seed, correct_dbn=False):
    m = EncounterModel(model_paths[model])
    ev = m.sample_events(n, T, seed=seed, device="cuda")
    ei, et = m.loglik_events(ev, correct_dbn=correct_dbn)
    ei, et = ei.cpu().numpy(), et.cpu().numpy()
    rows, off, ib = _host_rows(ev), ev.offsets.cpu().numpy(), ev.init_bins.cpu().numpy().T
    wi, wt = emu_events(EmuModel(model_paths[model]), ib, rows["dt"], rows["var"], rows["bin"], off, T, correct_dbn)
    assert np.array_equal(ei, wi), "initial term: device != host emulation"
    assert np.array_equal(et, wt), "transition term: device != host emulation"
    if len(m.gated_vars) <= 7 and T <= 1023:
        pk = m.sample_events_packed(n, T, seed=seed, device="cuda")
        pi, pt = m.loglik_events(pk, correct_dbn=correct_dbn)
        assert np.array_equal(pi.cpu().numpy(), ei) and np.array_equal(pt.cpu().numpy(), et), "packed rows score differently"
    tr = m.sample_tracks(n, T, seed=seed, device="cuda", want_values=False)
    di, dt = m.loglik_tracks(tr, correct_dbn=correct_dbn)
    di, dt = di.cpu().numpy(), dt.cpu().numpy()
    assert np.array_equal(ei, di), "initial term != dense scoring of the same tracks"
    if not m.is_dynvar_depend and not correct_dbn:
        assert np.array_equal(et, dt), "frozen transition term != dense scoring of the same tracks"
    else:
        assert_same(et, dt)
    assert np.isfinite(ei).all()
    return m, ev


def test_flagship_matches_emulation_and_dense_scoring(model_paths):
    """20 000 x 600 s of the flagship model, 8-byte and packed rows: frozen branch, bit for bit everywhere"""
    m, _ = _check(model_paths, UNCOR, 20_000, 600, seed=101)
    assert not m.is_dynvar_depend


@pytest.mark.parametrize("model,n,T", [("glider_v1", 5_000, 120), ("cor_v1", 3_000, 60), ("balloon_v1", 4_000, 50)])
def test_other_models(model_paths, model, n, T):
    _check(model_paths, model, n, T, seed=202)


@pytest.mark.parametrize("model", [UNCOR, "glider_v1"])
def test_correct_dbn(model_paths, model):
    _check(model_paths, model, 3_000, 99, seed=303, correct_dbn=True)


def test_host_buffers_equal_device_buffers(model_paths):
    m = EncounterModel(model_paths["cor_v1"])
    ev = m.sample_events(1_000, 37, seed=505, device="cuda")
    di, dt = m.loglik_events(ev)
    hi, ht = m.loglik_events(_host_rows(ev).copy(), ev.offsets.cpu().numpy(), 37, ev.init_bins.cpu().numpy())
    assert isinstance(hi, np.ndarray) and np.array_equal(hi, di.cpu().numpy()) and np.array_equal(ht, dt.cpu().numpy())
    pk = m.sample_events_packed(1_000, 37, seed=505, device="cuda")
    hi, ht = m.loglik_events(pk.words.cpu().numpy().view(np.uint32), pk.offsets.cpu().numpy(), 37, pk.init_bins.cpu().numpy(),
                             dts=pk.dts.cpu().numpy())
    assert np.array_equal(hi, di.cpu().numpy()) and np.array_equal(ht, dt.cpu().numpy())


def _refused(m, rows, off, ev, message, dts=None):
    with pytest.raises(L.EmbError) as ei:
        m.loglik_events(rows, off, ev.T, ev.init_bins, dts=dts)
    assert ei.value.code == L.EMB_E_ARG and message in ei.value.message, ei.value.message
    torch.cuda.synchronize()


def test_corrupted_rows_are_refused(model_paths):
    m = EncounterModel(model_paths[UNCOR])
    ev = m.sample_events(2_000, 120, seed=606, device="cuda")
    rows, off = _host_rows(ev).copy(), ev.offsets.cpu().numpy()
    ib = ev.init_bins.cpu().numpy()
    dyn = [int(v) for v in m.temporal_map[:, 0]]
    static = [v for v in range(1, m.n_initial + 1) if v not in dyn]
    k = int(np.nonzero(np.isin(rows["var"], dyn))[0][50])                  # a real row of a dynamic variable
    s = int(np.searchsorted(off, k, side="right") - 1)                      # its track

    def dev(r, o=off):
        return torch.from_numpy(np.ascontiguousarray(r).view(np.int64)).cuda(), torch.from_numpy(np.ascontiguousarray(o)).cuda()

    bad = rows.copy()
    bad["bin"][k] = 99
    _refused(m, *dev(bad), ev, "outside 1..r")
    bad = rows.copy()
    bad["var"][k] = m.n_initial + 1
    _refused(m, *dev(bad), ev, "variable id is outside 0..n_initial")
    bad = rows.copy()
    v = static[0]
    bad["var"][k], bad["bin"][k] = v, ib[v - 1, s] % m.r_initial[v - 1] + 1
    _refused(m, *dev(bad), ev, "static variable")
    # a row at column 0 after the track's other column-0 rows, setting a dynamic variable to another bin
    j = int(off[s]) + int(np.argmax(rows["dt"][off[s]:off[s + 1]] > 0))
    row = np.zeros(1, dtype=L.EVENT_DTYPE)
    row["var"], row["bin"] = dyn[0], ib[dyn[0] - 1, s] % m.r_initial[dyn[0] - 1] + 1
    bad, boff = np.insert(rows, j, row), off.copy()
    boff[s + 1:] += 1
    _refused(m, *dev(bad, boff), ev, "column 0")
    boff = off.copy()
    boff[10] = boff[11] + 1
    _refused(m, *dev(rows, boff), ev, "offsets must be non-negative and non-decreasing")
    # packed rows: a gated ordinal above n_gated, and a bin above r
    pk = m.sample_events_packed(2_000, 120, seed=606, device="cuda")
    w = pk.words.cpu().numpy().view(np.uint32).copy()
    kp = int(np.nonzero((w >> 27) & 7)[0][50])
    if len(m.gated_vars) < 7:
        bw = w.copy()
        bw[kp] = (bw[kp] & ~np.uint32(7 << 27)) | np.uint32(7 << 27)
        _refused(m, torch.from_numpy(bw.view(np.int32)).cuda(), pk.offsets, pk, "gated ordinal above n_gated", dts=pk.dts)
    g = int((w[kp] >> 27) & 7)
    if m.r_initial[m.gated_vars[g - 1] - 1] < 16:
        bw = w.copy()
        bw[kp] |= np.uint32(15 << 23)
        _refused(m, torch.from_numpy(bw.view(np.int32)).cuda(), pk.offsets, pk, "outside 1..r", dts=pk.dts)
    # the device is still usable and the real rows still score
    i, t = m.loglik_events(ev)
    assert torch.isfinite(i).all() and torch.isfinite(t).all()


def test_flagship_at_scale_packed(model_paths):
    """1.25M x 600 s, device-resident packed rows: the dense scoring of the same seed, bit for bit (frozen branch)"""
    m = EncounterModel(model_paths[UNCOR])
    n, T = 1_250_000, 600
    pk = m.sample_events_packed(n, T, seed=707, device="cuda", want_init=True)
    ei, et = m.loglik_events(pk)
    del pk
    tr = m.sample_tracks(n, T, seed=707, device="cuda", want_values=False)
    di, dt = m.loglik_tracks(tr)
    assert torch.equal(ei, di) and torch.equal(et, dt)
    assert torch.isfinite(et).all()
