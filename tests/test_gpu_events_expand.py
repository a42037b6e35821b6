"""GPU suite for out_samples and control rows from event lists (`-m gpu`, on the B200): k_events_expand on the rows of
sample_events and sample_events_packed against the host emulation of the same code bit for bit, with device and host buffers;
sample_batch against UncorEncounterModel.sample; the capacity protocol; one flagship run of 1.25M x 600 s; the status-word
refusals on corrupted copies of real rows."""
import ctypes as C

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from test_events_expand import EmuModel, assert_bits, emu_expand

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

UNCOR = "uncor_allcode_fwsingle_v1"


def _flat(ctl):
    return np.concatenate(ctl, axis=0) if ctl else np.zeros((0, 1))


def _check_result(em, res, T, packed, spec=None):
    """device buffers and host buffers against the emulation, for one sampled event result"""
    m = em.m
    smp, ctl = m.expand_events_gpu(res, spec=spec)
    off = res.offsets.cpu().numpy()
    iv = res.init_values.cpu().numpy()
    if packed:
        rows, dts = res.words.cpu().numpy().view(np.uint32), res.dts.cpu().numpy()
    else:
        rows, dts = res.events.cpu().numpy().view(L.EVENT_DTYPE), None
    ws, wc = emu_expand(em, iv.T, rows, dts, off, T, packed=packed, spec=spec)
    assert_bits(smp.cpu().numpy(), ws, "device samples vs emulation")
    assert np.array_equal(ctl.offsets.cpu().numpy()[1:] - ctl.offsets.cpu().numpy()[:-1], [len(c) for c in wc])
    assert_bits(ctl.rows.cpu().numpy(), _flat(wc), "device controls vs emulation")
    hs, hc = m.expand_events_gpu(rows, off, T, iv, dts=dts, spec=spec)       # host buffers, staged by the library
    assert_bits(hs, ws, "host-buffer samples vs emulation")
    assert_bits(hc.rows, _flat(wc), "host-buffer controls vs emulation")
    assert np.array_equal(hc.offsets, ctl.offsets.cpu().numpy())


@pytest.mark.parametrize("model,n,T,uncor", [(UNCOR, 3_000, 600, True), ("glider_v1", 3_000, 120, True),
                                             ("cor_v1", 2_000, 60, False), ("balloon_v1", 2_000, 50, False)])
def test_device_equals_emulation(model_paths, model, n, T, uncor):
    em = EmuModel(model_paths[model], idx_zero=(1, 2, 3) if uncor else (), uncor=uncor)
    m = em.m
    spec = m.out_eme_spec() if uncor and m.idxDH and m.idxDPsi and m.idxDV else None
    _check_result(em, m.sample_events(n, T, seed=11, device="cuda"), T, packed=False)
    _check_result(em, m.sample_events(n, T, seed=12, device="cuda"), T, packed=False, spec=spec)
    if len(m.gated_vars) <= 7 and T <= 1023:
        _check_result(em, m.sample_events_packed(n, T, seed=13, device="cuda"), T, packed=True)
        _check_result(em, m.sample_events_packed(n, T, seed=14, device="cuda"), T, packed=True, spec=spec)


def test_sample_batch_equals_sample(model_paths):
    """packed=False reads the same fp32 row values as UncorEncounterModel.sample: out_samples and out_EME.event bit for bit"""
    m = EmuModel(model_paths[UNCOR], idx_zero=(1, 2, 3), uncor=True).m
    n, T = 300, 600
    oi, oe, osmp, oeme = m.sample(n, T, seed=77)
    for device in (None, "cuda"):
        bi, res, smp, ctl = m.sample_batch(n, T, seed=77, packed=False, want_samples=True, device=device)
        if device is not None:
            bi, smp = bi.cpu().numpy(), smp.cpu().numpy()
            ctl.rows, ctl.offsets = ctl.rows.cpu().numpy(), ctl.offsets.cpu().numpy()
        assert_bits(bi, oi, "out_inits")
        for s in range(n):
            assert_bits(smp[s].T, osmp[s], "out_samples{%d}" % s)
            assert_bits(ctl.track(s), oeme[s].event, "out_EME(%d).event" % s)
    _, pres, psmp, pctl = m.sample_batch(n, T, seed=77, want_samples=True)     # packed rows: the same lists, fp64 values
    assert np.array_equal(pctl.offsets, ctl.offsets)
    assert_bits(pctl.rows[:, 0], ctl.rows[:, 0], "control times of packed and 8-byte rows")


def test_capacity_protocol(model_paths):
    m = EmuModel(model_paths[UNCOR], idx_zero=(1, 2, 3), uncor=True).m
    n, T = 500, 600
    res = m.sample_events_packed(n, T, seed=5)
    iv = np.ascontiguousarray(res.init_values)
    lib, o = L.lib(), m._opts()
    cs = L.ControlsSpec()
    total = C.c_int64(-1)
    off = np.full(n + 1, -7, dtype=np.int64)
    smp = np.full(n * T * m.n_initial, 1.25)
    ctl = np.full(1, 2.5)

    def call(capacity, rows):
        return lib.emb_track_events_expand_packed(m._h, n, T, iv.ctypes.data, res.words.ctypes.data, res.dts.ctypes.data,
                                                  res.offsets.ctypes.data, C.byref(o), C.byref(cs), smp.ctypes.data, capacity,
                                                  None if rows is None else rows.ctypes.data, off.ctypes.data, C.byref(total))

    assert call(0, None) == L.EMB_E_LIMIT and "rows needed" in lib.emb_last_error().decode()
    need = total.value
    assert need > 0 and off[0] == 0 and off[n] == need and np.all(np.diff(off) > 0)
    assert np.all(smp == 1.25), "samples written by a sizing call"
    rows = np.full((need - 1, 1 + m.n_dyn), 2.5)
    assert call(need - 1, rows) == L.EMB_E_LIMIT and total.value == need
    assert np.all(rows == 2.5) and np.all(smp == 1.25), "outputs written although the buffer was too small"
    rows = np.full((need, 1 + m.n_dyn), 2.5)
    assert call(need, rows) == 0 and total.value == need
    ws, wc = m.expand_events_gpu(res)
    assert_bits(smp.reshape(n, T, m.n_initial), ws, "samples after the retry")
    assert_bits(rows, wc.rows, "controls after the retry")
    assert np.array_equal(off, wc.offsets)
    del ctl


def test_flagship_controls_1p25m(model_paths):
    """1.25M x 600 s packed rows to the out_EME rows on the device; 300 tracks spot-checked against the emulation"""
    em = EmuModel(model_paths[UNCOR], idx_zero=(1, 2, 3), uncor=True)
    m = em.m
    n, T = 1_250_000, 600
    out_inits, res, smp, ctl = m.sample_batch(n, T, seed=2024, device="cuda")
    assert smp is None and ctl.rows.shape[1] == 4
    off, coff = res.offsets.cpu().numpy(), ctl.offsets.cpu().numpy()
    assert coff[n] == ctl.rows.shape[0] > n
    pick = np.sort(np.random.default_rng(1).choice(n, 300, replace=False))
    parts = [np.arange(off[s], off[s + 1]) for s in pick]
    idx = torch.from_numpy(np.concatenate(parts)).cuda()
    words, dts = res.words[idx].cpu().numpy().view(np.uint32), res.dts[idx].cpu().numpy()
    noff = np.concatenate(([0], np.cumsum([len(q) for q in parts]))).astype(np.int64)
    iv = out_inits[torch.from_numpy(pick).cuda()].cpu().numpy()
    _, wc = emu_expand(em, iv, words, dts, noff, T, packed=True, spec=m.out_eme_spec(), samples=False)
    rows = ctl.rows.cpu().numpy()
    for k, s in enumerate(pick):
        assert_bits(rows[coff[s]:coff[s + 1]], wc[k], "track %d" % s)


def test_corrupted_rows_are_refused(model_paths):
    m = EmuModel(model_paths[UNCOR], idx_zero=(1, 2, 3), uncor=True).m
    n, T = 200, 600
    pk = m.sample_events_packed(n, T, seed=31, device="cuda")
    words = pk.words.clone()
    k = int(torch.nonzero((words >> 27) & 7 > 0)[5])
    words[k] = (words[k] & ~(15 << 23)) | (15 << 23)                           # bin 16: above r of every gated variable
    with pytest.raises(L.EmbError) as ei:
        m.expand_events_gpu(words, pk.offsets, T, pk.init_values, dts=pk.dts)
    assert ei.value.code == L.EMB_E_ARG and "bin is outside 1..r" in ei.value.message
    ev = m.sample_events(n, T, seed=31, device="cuda")
    rows = ev.events.clone().view(torch.uint8).view(-1, 8)
    rows[7, 2] = 200                                                            # variable id 200
    with pytest.raises(L.EmbError) as ei:
        m.expand_events_gpu(rows.view(torch.int64).view(-1), ev.offsets, T, ev.init_values)
    assert ei.value.code == L.EMB_E_ARG and "variable id" in ei.value.message
    off = ev.offsets.clone()
    off[3] = off[5] + 1                                                         # decreasing
    with pytest.raises(L.EmbError) as ei:
        m.expand_events_gpu(ev.events, off, T, ev.init_values)
    assert ei.value.code == L.EMB_E_ARG and "offsets" in ei.value.message
