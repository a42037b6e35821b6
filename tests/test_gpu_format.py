"""GPU suite for the em_sample text formatter (`-m gpu`, on the B200): k_format_{initial,transition}[_count] through
emb_format_em_sample on crafted arrays, with host and device buffers, against Python's '%g' rows and the host emulation; em_sample
files byte-identical to the host formatting loop it replaced on the same sample_tracks output; the capacity protocol; the
refusals."""
import ctypes as C

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel, tile
from test_format import emu_text, rows_initial, rows_transition

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _dyn_cols(m):
    tv = list(m.timevarying_vars)
    return [tv.index(int(v)) for v in m.temporal_map[:, 0]]


def _crafted(m, n, T, seed):
    rng = np.random.default_rng(seed)
    iv = rng.standard_normal((m.n_initial, n)) * 10.0 ** rng.integers(-8, 9, (m.n_initial, n))
    iv.flat[:6] = [-0.0, 0.0, 999999.5, 9.999995e-05, 5e-324, 1.7976931348623157e308][:iv.size]
    vals = (rng.standard_normal((n, len(m.timevarying_vars), T)) * 10.0 ** rng.integers(-6, 7, (n, len(m.timevarying_vars), T)))
    return iv, vals.astype(np.float32)


@pytest.mark.parametrize("n,T,first_id", [(1, 1, 1), (300, 7, 999_901), (129, 60, 1), (257, 5, 2 ** 53 - 257)])
def test_crafted_arrays_host_and_device(model_paths, n, T, first_id):
    m = EncounterModel(model_paths["cor_v1"])
    iv, vals = _crafted(m, n, T, n + T)
    vt = tile(vals)
    want_i = rows_initial(iv, first_id).encode()
    want_t = rows_transition(vals[:, _dyn_cols(m), :].astype(np.float64), first_id).encode()
    emu_i, emu_io = emu_text(n, T, first_id, m.n_initial, _dyn_cols(m), len(m.timevarying_vars), iv, None, False)
    emu_t, emu_to = emu_text(n, T, first_id, m.n_initial, _dyn_cols(m), len(m.timevarying_vars), None, vt, True)
    assert emu_i == want_i and emu_t == want_t
    host = m.format_em_sample(iv, vt, T, first_id=first_id)
    dev = m.format_em_sample(torch.from_numpy(iv).cuda(), torch.from_numpy(vt).cuda(), T, first_id=first_id)
    for ti, oi, tt, ot in (host, dev):
        assert _np(ti).tobytes() == want_i and _np(tt).tobytes() == want_t
        assert np.array_equal(_np(oi), emu_io) and np.array_equal(_np(ot), emu_to)
    # either text alone
    ti, oi, tt, ot = m.format_em_sample(iv, None, T, first_id=first_id)
    assert ti.tobytes() == want_i and tt is None and ot is None
    ti, oi, tt, ot = m.format_em_sample(None, vt, T, first_id=first_id, n=n)
    assert ti is None and tt.tobytes() == want_t


def _host_loop(m, res, first):
    """the formatting loop of em_sample.py before the device formatter, on the same sample_tracks output"""
    iv = _np(res.init_values)
    vals = np.asarray(_np(res.values), dtype=np.float64)[:, _dyn_cols(m), :]
    return rows_initial(iv, first + 1).encode(), rows_transition(vals, first + 1).encode()


@pytest.mark.parametrize("model", ["cor_v1", "uncor_1200code_v2p1"])
@pytest.mark.parametrize("n,T,chunk", [(300, 7, 1 << 16), (5, 1, 1 << 16), (400, 60, 128), (1000, 13, 384)])
def test_em_sample_files_match_host_loop(model_paths, tmp_path, model, n, T, chunk):
    from em_model_manned_bayes_b200.em_sample import em_sample
    fi, ft = str(tmp_path / "initial.txt"), str(tmp_path / "transition.txt")
    em_sample(model_paths[model], fi, ft, num_initial_samples=n, num_transition_samples=T, rng_seed=42, chunk=chunk)
    m = EncounterModel(model_paths[model], idxZeroBoundaries=(1, 2, 3))
    want_i = ("id " + "".join("%s " % l for l in m.labels_initial) + "\n").encode()
    want_t = ("initial_id t " + "".join("%s " % m.labels_transition[int(k) - 1] for k in m.temporal_map[:, 1]) + "\n").encode()
    for first in range(0, n, chunk):
        res = m.sample_tracks(min(chunk, n - first), T, seed=42, first_sample=first, want_bins=False)
        a, b = _host_loop(m, res, first)
        want_i += a
        want_t += b
    assert open(fi, "rb").read() == want_i
    assert open(ft, "rb").read() == want_t


def _opts(mem=L.EMB_MEM_HOST):
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem = mem
    return o


def test_capacity_protocol(model_paths):
    m = EncounterModel(model_paths["uncor_1200code_v2p1"])
    n, T = 200, 9
    res = m.sample_tracks(n, T, seed=3, device="cuda")
    ti, oi, tt, ot = m.format_em_sample(res, first_id=11)
    lib = L.lib()
    o = _opts(L.EMB_MEM_DEVICE)
    iv, vt = res.init_values.contiguous(), res.values_tiled.contiguous()
    off_i = torch.full((n + 1,), -1, dtype=torch.int64, device="cuda")
    off_t = torch.full((n + 1,), -1, dtype=torch.int64, device="cuda")
    buf_i = torch.zeros(len(ti), dtype=torch.uint8, device="cuda")
    buf_t = torch.zeros(len(tt) - 1, dtype=torch.uint8, device="cuda")     # one byte short
    totals = (C.c_int64 * 2)()
    rc = lib.emb_format_em_sample(m._h, n, T, 11, iv.data_ptr(), vt.data_ptr(), C.byref(o), len(ti), buf_i.data_ptr(),
                                  off_i.data_ptr(), len(tt) - 1, buf_t.data_ptr(), off_t.data_ptr(), totals)
    assert rc == L.EMB_E_LIMIT
    assert (totals[0], totals[1]) == (len(ti), len(tt))
    assert torch.equal(off_i, oi) and torch.equal(off_t, ot)
    assert int(buf_i.count_nonzero()) == 0 and int(buf_t.count_nonzero()) == 0       # no text written
    buf_t = torch.zeros(len(tt), dtype=torch.uint8, device="cuda")
    rc = lib.emb_format_em_sample(m._h, n, T, 11, iv.data_ptr(), vt.data_ptr(), C.byref(o), len(ti), buf_i.data_ptr(),
                                  off_i.data_ptr(), len(tt), buf_t.data_ptr(), off_t.data_ptr(), totals)
    assert rc == 0
    assert torch.equal(buf_i, ti) and torch.equal(buf_t, tt)
    # n = 0, host and device offsets
    for mem, dev in ((L.EMB_MEM_HOST, None), (L.EMB_MEM_DEVICE, "cuda")):
        off = np.full(1, -1, dtype=np.int64) if dev is None else torch.full((1,), -1, dtype=torch.int64, device=dev)
        ptr = off.ctypes.data if dev is None else off.data_ptr()
        rc = lib.emb_format_em_sample(m._h, 0, T, 1, None, None, C.byref(_opts(mem)), 0, None, ptr, 0, None, None, totals)
        assert rc == 0 and int(off[0]) == 0 and (totals[0], totals[1]) == (0, 0)


def test_refusals(model_paths):
    m = EncounterModel(model_paths["cor_v1"])
    n, T = 40, 6
    iv, vals = _crafted(m, n, T, 1)
    for bad in (np.inf, -np.inf, np.nan):
        iv2 = iv.copy()
        iv2[3, 17] = bad
        with pytest.raises(L.EmbError) as ei:
            m.format_em_sample(torch.from_numpy(iv2).cuda(), None, T)
        assert ei.value.code == L.EMB_E_ARG and "finite" in str(ei.value)
        vals2 = vals.copy()
        vals2[5, _dyn_cols(m)[1], 4] = bad
        with pytest.raises(L.EmbError) as ei:
            m.format_em_sample(None, tile(vals2), T, n=n)
        assert ei.value.code == L.EMB_E_ARG
    vt = tile(vals)
    with pytest.raises(L.EmbError) as ei:
        m.format_em_sample(iv, vt, T, first_id=0)
    assert ei.value.code == L.EMB_E_ARG
    with pytest.raises(L.EmbError) as ei:
        m.format_em_sample(iv, vt, T, first_id=2 ** 53 - n + 1)
    assert ei.value.code == L.EMB_E_ARG and "2^53" in str(ei.value)
    m.format_em_sample(iv, vt, T, first_id=2 ** 53 - n)
    o = _opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)
    off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_iv = torch.from_numpy(iv).cuda()
    rc = L.lib().emb_format_em_sample(m._h, n, T, 1, d_iv.data_ptr(), None, C.byref(o), 0, None, off.data_ptr(), 0, None, None, None)
    assert rc == L.EMB_E_ARG and "EMB_MEM_ASYNC" in L.lib().emb_last_error().decode()
    t = EncounterModel(model_paths["terminal_v3_radar_encounter_model"])   # no transition network
    tiv = np.ones((t.n_initial, 3))
    vt = np.zeros(16, np.float32)
    toff = np.zeros(4, dtype=np.int64)
    rc = L.lib().emb_format_em_sample(t._h, 3, 2, 1, tiv.ctypes.data, vt.ctypes.data, C.byref(_opts()), 0, None, None, 0, None,
                                      toff.ctypes.data, None)
    assert rc == L.EMB_E_ARG and "dynvar:empty" in L.lib().emb_last_error().decode()
    ti, _, tt, _ = t.format_em_sample(tiv, None, 2)                    # the initial text needs no transition network
    assert tt is None and ti.tobytes() == "".join("%d" % (s + 1) + " 1" * t.n_initial + "\n" for s in range(3)).encode()
