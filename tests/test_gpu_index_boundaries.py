"""GPU suite (`-m gpu`): sampling where the global sample index or the call size crosses an edge of the kernels.

Counter word 0 of the step stream is `sample >> 32` (stream spec v5), which the specialised track kernel treats as uniform
over a launch, so `launch_tracks` cuts a call at every multiple of 2^32 (`next_segment`).  Here every path that runs that
cut is checked on the device against an independent reference: the plain-C oracle (oracle/oracle_c.c), the Python oracle,
the host emulation (tests/emu) and numpy -- the dense tracks of every model shape with both kernels, the padding of the
last tile, the event passes (single pass and host pipeline), the fused integration, the initial network (whose call table
changes with `sample >> 34`), the multi-device shards and the terminal chains.  The size edges are the prefix sum of the
event rows past 1024 tiles of 2048 tracks, and an event list of more than 2^31 rows."""
import ctypes as C

import numpy as np
import pytest

import cases
import helpers as H
from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import CorTerminalModel, EncounterModel, TrackResult, UncorEncounterModel
from oracle.em_read import em_read
from test_gpu_parity import SWEEP

pytestmark = pytest.mark.gpu

B32, B34 = 2 ** 32, 2 ** 34
_ORACLE = {}


def _c_oracle(model_paths, model, uncor, n, T, seed, first):
    """COracle.sample_tracks, cached: both kernels are compared with the same reference"""
    from oracle.c_oracle import COracle
    key = (model, uncor, n, T, seed, first)
    if key not in _ORACLE:
        ref = COracle(em_read(model_paths[model]), uncor=uncor).sample_tracks(n, T, seed=seed, first_sample=first, threads=0)
        assert ref["rc"] == 0
        _ORACLE[key] = ref
    return _ORACLE[key]


class _generic:
    """force the generic kernels inside the block (or not)"""

    def __init__(self, on):
        self.on = int(on)

    def __enter__(self):
        L.lib().emb_debug_force_generic(self.on)

    def __exit__(self, *a):
        L.lib().emb_debug_force_generic(0)


def _model(model_paths, model, uncor):
    return (UncorEncounterModel if uncor else EncounterModel)(model_paths[model])


def _opts(m, uncor, **kw):
    return m.uncor_opts(**kw) if uncor else m._opts()


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _emu_opts(p, uncor=True, **kw):
    if uncor:
        lab = p.labels_initial
        kw.update(reject_mode=L.EMB_REJECT_UNCOR, idx_v=cases.label_index(lab, '"v"'),
                  idx_dh=cases.label_index(lab, '"\\dot h"'), idx_L=cases.label_index(lab, '"L"'))
    return H.EmuModel.opts(p.n_initial, **kw)


def _dyn_tv(p):
    dyn = [int(v) - 1 for v in np.asarray(p.temporal_map)[:, 0]]
    rates = np.asarray(p.resample_rates)
    return dyn, sorted(set(dyn) | {i for i in range(p.n_initial) if rates[i] > 0})


def _check_against_oracle(got, ref, p, where):
    dyn, tv = _dyn_tv(p)
    assert np.array_equal(_np(got.init_bins).T, ref["init_bins"]), where + ": initial bins"
    assert np.array_equal(_np(got.attempts).astype(np.int64), ref["attempts"].astype(np.int64)), where + ": attempts"
    assert np.array_equal(_np(got.init_values).T, ref["init_values"]), where + ": initial values"
    assert np.array_equal(_np(got.bins), ref["sample_bins"][:, dyn, :]), where + ": dense bins"
    want = ref["samples"][:, tv, :]
    assert np.all(np.abs(_np(got.values).astype(np.float64) - want) <= 1e-6 * np.abs(want)), where + ": dense values"


def _full(buf, nvar, n, T):
    """the whole tiled buffer as (128 * ceil(n/128), nvar, 4 * ceil(T/4)), padding tracks and seconds included"""
    a = _np(buf)
    nch, ntile = (T + 3) // 4, (n + 127) // 128
    return a.reshape(nch, ntile, nvar, 128, 4).transpose(1, 3, 2, 0, 4).reshape(ntile * 128, nvar, nch * 4)


# ---- A. dense tracks across 2^32 ------------------------------------------------------------------------------------
# (k, o): first_sample = k * 2^32 - o, i.e. o tracks before the boundary: one track in, mid-tile, either side of a tile edge
CUTS = [(1, 1), (2, 37), (3, 127), (5, 128), (0xFFFF, 200)]
N_A, T_A = 333, 45


@pytest.mark.parametrize("generic", [0, 1], ids=["specialised", "generic"])
@pytest.mark.parametrize("model,uncor", [(s[0], s[1]) for s in SWEEP])
def test_tracks_across_2_32_match_c_oracle(model_paths, model, uncor, generic):
    """Every model shape, both kernels: a call that straddles a multiple of 2^32 equals the C oracle (bins, attempts and
    initial values exact, dense values within 1e-6), and host buffers equal device buffers byte for byte, padding included."""
    p = em_read(model_paths[model])
    m = _model(model_paths, model, uncor)
    for k, o in CUTS:
        first = k * B32 - o
        ref = _c_oracle(model_paths, model, uncor, N_A, T_A, 31, first)
        with _generic(generic):
            dev = m.sample_tracks(N_A, T_A, seed=31, first_sample=first, opts=_opts(m, uncor), device="cuda:0")
            assert L.lib().emb_debug_last_kernel_fast() == (0 if generic else 1)
            host = m.sample_tracks(N_A, T_A, seed=31, first_sample=first, opts=_opts(m, uncor))
        _check_against_oracle(dev, ref, p, "%s o=%d" % (model, o))
        for a, b in ((host.bins_tiled, dev.bins_tiled), (host.values_tiled, dev.values_tiled), (host.init_bins, dev.init_bins),
                     (host.init_values, dev.init_values), (host.attempts, dev.attempts)):
            assert np.array_equal(a.view(np.uint8), _np(b).view(np.uint8)), "%s o=%d: host != device" % (model, o)


@pytest.mark.parametrize("generic", [0, 1], ids=["specialised", "generic"])
def test_correct_dbn_across_2_32_matches_the_oracle(model_paths, generic):
    """correct_dbn (parents re-evaluated every second) across the boundary, against the Python oracle with the same option"""
    from oracle.drivers import uncor_sample
    from oracle.uniforms import KeyedPhilox
    p = em_read(model_paths["uncor_1200code_v2p1"])
    n, T, first = 40, 62, 4 * B32 - 23
    bins, vals, _, _ = H.oracle_dense(p, uncor_sample(p, n, T, KeyedPhilox(8), first_sample=first, correct_dbn=True))
    m = UncorEncounterModel(model_paths["uncor_1200code_v2p1"])
    with _generic(generic):
        got = m.sample_tracks(n, T, seed=8, first_sample=first, opts=m.uncor_opts(correct_dbn=True), device="cuda:0")
        assert L.lib().emb_debug_last_kernel_fast() == (0 if generic else 1)
    assert np.array_equal(_np(got.bins), bins)
    assert np.all(np.abs(_np(got.values).astype(np.float64) - vals) <= 1e-6 * np.abs(vals))


@pytest.mark.parametrize("generic", [0, 1], ids=["specialised", "generic"])
@pytest.mark.parametrize("model,uncor", [("uncor_1200code_v2p1", True), ("glider_v1", True), ("cor_v1", False)])
def test_histograms_across_2_32_count_the_oracle_bins(model_paths, model, uncor, generic):
    """Each launch of a split call flushes its own histograms: their sum is the bincount of the oracle's bins."""
    import torch
    p = em_read(model_paths[model])
    m = _model(model_paths, model, uncor)
    first = 2 * B32 - 200
    ref = _c_oracle(model_paths, model, uncor, N_A, T_A, 31, first)
    hi =torch.zeros((m.n_initial, 64), dtype=torch.int64, device="cuda:0")
    ht = torch.zeros((m.n_dyn, 64), dtype=torch.int64, device="cuda:0")
    with _generic(generic):
        got = m.sample_tracks(N_A, T_A, seed=31, first_sample=first, opts=_opts(m, uncor), device="cuda:0",
                              hist_initial=hi, hist_transition=ht)
    _check_against_oracle(got, ref, p, model)
    dyn, _ = _dyn_tv(p)
    for i in range(m.n_initial):
        assert np.array_equal(_np(hi[i]), np.bincount(ref["init_bins"][:, i].astype(np.int64) - 1, minlength=64)), ("initial", i)
    for d, v in enumerate(dyn):
        want = np.bincount(ref["sample_bins"][:, v, 1:].reshape(-1).astype(np.int64) - 1, minlength=64)
        assert np.array_equal(_np(ht[d]), want), ("transition", d)


# ---- B. padding tracks and seconds -----------------------------------------------------------------------------------
# (first_sample, n): split with padding, split at a tile edge, a boundary one track in, and two calls without a split
PAD_GRID = [(B32 - 1, 129), (B32 - 100, 300), (B32 - 37, 300), (3 * B32 - 200, 250), (B32 - 128, 200), (B32 - 64, 128), (B32 - 1, 1),
            (B32 - 300, 129), (5, 129)]
T_B = 45


def _sentinel_tracks(m, n, T):
    import torch
    nb, nv = int(L.lib().emb_tracks_bins_len(m._h, n, T)), int(L.lib().emb_tracks_values_len(m._h, n, T))
    ni = m.n_initial
    dev = "cuda:0"
    return TrackResult(n=n, T=T, dyn_vars=[int(v) for v in m.temporal_map[:, 0]], tv_vars=list(m.timevarying_vars),
                       bins_tiled=torch.full((nb,), -1, dtype=torch.int8, device=dev),
                       values_tiled=torch.full((nv,), float("nan"), dtype=torch.float32, device=dev),
                       init_bins=torch.full((ni, n), -1, dtype=torch.int8, device=dev),
                       init_values=torch.full((ni, n), float("nan"), dtype=torch.float64, device=dev),
                       attempts=torch.full((n,), -1, dtype=torch.int16, device=dev))


def _check_padding(res, m, n, T, where):
    """padding tracks and padding seconds are 0; no real track kept the sentinel (-1 / NaN)"""
    b = _full(res.bins_tiled, m.n_dyn, n, T)
    v = _full(res.values_tiled, len(m.timevarying_vars), n, T)
    for name, a in (("bins", b), ("values", v)):
        assert not np.any(a[n:]), "%s: padding tracks of the %s are not 0 (%d nonzero)" % (where, name, int(np.count_nonzero(a[n:])))
        assert not np.any(a[:n, :, T:]), "%s: padding seconds of the %s are not 0" % (where, name)
    assert np.all(b[:n, :, :T] >= 1), where + ": a real track has bin < 1"
    assert not np.any(np.isnan(v[:n, :, :T])), where + ": a real track kept NaN"
    if res.init_bins is not None:
        assert np.all(_np(res.init_bins) >= 1) and not np.any(np.isnan(_np(res.init_values)))
        assert np.all(_np(res.attempts).astype(np.int64) >= 1)


@pytest.mark.parametrize("generic", [0, 1], ids=["specialised", "generic"])
def test_padding_tracks_are_zero_when_a_launch_is_split(model_paths, generic):
    """emb_sample_tracks into device buffers prefilled with -1 / NaN, and into host buffers staged from a memory pool that
    holds an earlier call's tracks: over first_sample mod 2^32 and n, every padding track and every padding second is 0."""
    m = UncorEncounterModel(model_paths["uncor_1200code_v2p1"])
    for first, n in PAD_GRID:
        where = "first=%d n=%d" % (first, n)
        with _generic(generic):
            res = _sentinel_tracks(m, n, T_B)
            m.sample_tracks(n, T_B, seed=3, first_sample=first, opts=m.uncor_opts(), device="cuda:0", out=res)
            _check_padding(res, m, n, T_B, where + " (device)")
            m.sample_tracks((n + 127) // 128 * 128, T_B, seed=4, opts=m.uncor_opts())      # fills the padding tracks' bytes
            host = m.sample_tracks(n, T_B, seed=3, first_sample=first, opts=m.uncor_opts())
        _check_padding(host, m, n, T_B, where + " (host)")
        assert np.array_equal(host.bins_tiled, _np(res.bins_tiled)) and np.array_equal(host.values_tiled, _np(res.values_tiled))


def test_padding_of_the_fused_xyz_dense_outputs(model_paths):
    """emb_sample_tracks_xyz with the dense outputs requested: the same zero padding, and the same tiles as emb_sample_tracks"""
    from em_model_manned_bayes_b200.sample2track import sample_tracks_xyz
    m = UncorEncounterModel(model_paths["uncor_1200code_v2p1"])
    for first, n in PAD_GRID:
        res = _sentinel_tracks(m, n, T_B)
        sample_tracks_xyz(m, n, T_B, seed=3, first_sample=first, sample_opts=m.uncor_opts(), device="cuda:0", dense=res)
        assert L.lib().emb_debug_last_kernel_fast() == 1
        _check_padding(res, m, n, T_B, "xyz first=%d n=%d" % (first, n))
        plain = m.sample_tracks(n, T_B, seed=3, first_sample=first, opts=m.uncor_opts(), device="cuda:0")
        assert np.array_equal(_np(res.bins_tiled), _np(plain.bins_tiled))
        assert np.array_equal(_np(res.values_tiled).view(np.uint32), _np(plain.values_tiled).view(np.uint32))


# ---- C. event lists across 2^32 -----------------------------------------------------------------------------------------
def _rows(ev):
    return _np(ev.events).view(L.EVENT_DTYPE) if not isinstance(ev.events, np.ndarray) else np.asarray(ev.events)


def _check_rows_equal_emu(rows, off, want, want_off, where):
    assert np.array_equal(_np(off), want_off), where + ": offsets"
    for f in ("dt", "var", "bin"):
        assert np.array_equal(rows[f], want[f]), where + ": " + f
    w = want["value"].astype(np.float64)
    assert np.all(np.abs(rows["value"].astype(np.float64) - w) <= 1e-6 * np.abs(w)), where + ": values"


def _joined(parts):
    """offsets and rows of calls over consecutive track ranges, joined as one call (offsets carried)"""
    off, rows, carry = [np.zeros(1, dtype=np.int64)], [], 0
    for o, r in parts:
        o = _np(o).astype(np.int64)
        off.append(o[1:] + carry)
        rows.append(r[:o[-1]])
        carry += int(o[-1])
    return np.concatenate(off), np.concatenate(rows)


@pytest.mark.parametrize("generic", [0, 1], ids=["specialised", "generic"])
def test_device_event_lists_across_2_32(model_paths, generic):
    """Device-resident single pass (count -> scan -> write), 8-byte and packed rows, across 2^32: rows equal the host
    emulation, the packed rows decode to the Python oracle's fp64 values on the tracks around the boundary, and the offsets
    equal those of the same tracks sampled in two calls that do not cross it."""
    from oracle.drivers import uncor_sample
    from oracle.uniforms import KeyedPhilox
    name = "uncor_1200code_v2p1"
    p = em_read(model_paths[name])
    m = UncorEncounterModel(model_paths[name])
    n, T, b = 700, 90, 301
    first = 6 * B32 - b
    want, want_off = H.EmuModel(model_paths[name]).sample_events(n, T, 12, first, _emu_opts(p))
    with _generic(generic):
        ev = m.sample_events(n, T, seed=12, first_sample=first, opts=m.uncor_opts(), device="cuda:0")
        assert L.lib().emb_debug_last_kernel_fast() == (0 if generic else 1)
        pk = m.sample_events_packed(n, T, seed=12, first_sample=first, opts=m.uncor_opts(), device="cuda:0")
        parts = [m.sample_events(k, T, seed=12, first_sample=f, opts=m.uncor_opts(), device="cuda:0")
                 for f, k in ((first, b), (first + b, n - b))]
    rows = _rows(ev)
    _check_rows_equal_emu(rows, ev.offsets, want, want_off, "8-byte rows")
    assert ev.total == int(want_off[-1])
    joff, jrows = _joined([(q.offsets, _rows(q)) for q in parts])
    assert np.array_equal(joff, want_off) and np.array_equal(jrows.view(np.int64), rows.view(np.int64))
    dt, var, binv, val = pk.decode()
    assert np.array_equal(_np(pk.offsets), want_off) and pk.total == ev.total
    assert np.array_equal(dt, rows["dt"]) and np.array_equal(var, rows["var"]) and np.array_equal(binv, rows["bin"])
    assert np.all(np.abs(val - rows["value"]) <= 1e-6 * np.abs(val))
    # fp64 event values of the Python oracle on the tracks either side of the boundary
    lo, hi = b - 6, b + 6
    ref = uncor_sample(p, hi - lo, T, KeyedPhilox(12), first_sample=first + lo)
    a, z = int(want_off[lo]), int(want_off[hi])
    ref_ev = np.concatenate([s.events for s in ref])
    assert np.array_equal(np.asarray(_np(ev.init_values))[:, lo:hi].T, np.stack([s.initial for s in ref]))
    assert ref_ev.shape[0] == z - a
    assert np.array_equal(dt[a:z], ref_ev[:, 0]) and np.array_equal(var[a:z], ref_ev[:, 1])
    assert np.all(np.abs(val[a:z] - ref_ev[:, 2]) <= 1e-12 * np.abs(ref_ev[:, 2]))


def test_host_pipelined_event_lists_across_2_32(model_paths):
    """Host buffers and n >= 8192: the chunked pipeline, with the boundary inside chunk 3 (not at a chunk edge), 8-byte and
    packed rows, against the host emulation and against two calls that do not cross the boundary."""
    name = "uncor_1200code_v2p1"
    p = em_read(model_paths[name])
    m = UncorEncounterModel(model_paths[name])
    n, T, b = 10_000, 60, 4321                 # chunk 3 holds tracks [3750, 5000)
    first = 2 * B32 - b
    want, want_off = H.EmuModel(model_paths[name]).sample_events(n, T, 13, first, _emu_opts(p))
    h = m.sample_events(n, T, seed=13, first_sample=first, opts=m.uncor_opts())
    _check_rows_equal_emu(np.asarray(h.events), h.offsets, want, want_off, "pipelined 8-byte rows")
    hp = m.sample_events_packed(n, T, seed=13, first_sample=first, opts=m.uncor_opts())
    dt, var, binv, _ = hp.decode()
    assert np.array_equal(hp.offsets, want_off)
    assert np.array_equal(dt, want["dt"]) and np.array_equal(var, want["var"]) and np.array_equal(binv, want["bin"])
    parts = [m.sample_events(k, T, seed=13, first_sample=f, opts=m.uncor_opts()) for f, k in ((first, b), (first + b, n - b))]
    joff, jrows = _joined([(q.offsets, np.asarray(q.events)) for q in parts])
    assert np.array_equal(joff, want_off) and np.array_equal(jrows.view(np.int64), np.asarray(h.events).view(np.int64))
    assert np.array_equal(np.asarray(h.init_values), np.concatenate([q.init_values for q in parts], axis=1))


def test_long_tracks_with_2_byte_dts_across_2_32(model_paths):
    """T > 1023: the 8-byte entry point switches the device rows to 2-byte dts; across 2^32 the rows equal the emulation."""
    name = "uncor_1200code_v2p1"
    p = em_read(model_paths[name])
    m = UncorEncounterModel(model_paths[name])
    n, T, b = 300, 1100, 129
    first = B32 - b
    want, want_off = H.EmuModel(model_paths[name]).sample_events(n, T, 14, first, _emu_opts(p))
    for generic in (0, 1):
        with _generic(generic):
            ev = m.sample_events(n, T, seed=14, first_sample=first, opts=m.uncor_opts(), device="cuda:0")
        rows = _rows(ev)
        _check_rows_equal_emu(rows, ev.offsets, want, want_off, "T=1100 generic=%d" % generic)
        assert np.array_equal(np.add.reduceat(rows["dt"].astype(np.int64), want_off[:-1]), np.full(n, T))


# ---- D. fused xyz, initial network, multi-device, terminal chains ---------------------------------------------------
def test_fused_xyz_across_2_32_equals_sample_then_integrate(model_paths):
    import torch
    from em_model_manned_bayes_b200.sample2track import integrate_tracks, sample_tracks_xyz
    for name, n, T in (("uncor_1200code_v2p1", 700, 91), ("glider_v1", 400, 63)):
        m = UncorEncounterModel(model_paths[name])
        first = 7 * B32 - 333
        res = m.sample_tracks(n, T, seed=15, first_sample=first, opts=m.uncor_opts(), device="cuda:0")
        xyz, good = integrate_tracks(m, res, device="cuda:0")
        fx, fg = sample_tracks_xyz(m, n, T, seed=15, first_sample=first, sample_opts=m.uncor_opts(), device="cuda:0")
        assert L.lib().emb_debug_last_kernel_fast() == 1
        assert torch.equal(fx, xyz) and torch.equal(fg, good), name


NARROW = "RTCA228_A3"      # terminal geometry: speed limits 68..186 ft/s reject most first draws


def _initial_ref(model_paths, model, n, seed, first, box):
    from oracle.c_oracle import COracle
    p = em_read(model_paths[model])
    b = None
    if box:
        lo, hi = np.full(p.n_initial, -np.inf), np.full(p.n_initial, np.inf)
        for lab in ('"own_speed"', '"int_speed"'):
            lo[p.labels_initial.index(lab)], hi[p.labels_initial.index(lab)] = CorTerminalModel.DYN_LIMITS[NARROW]
        b = (lo, hi)
    r = COracle(p).sample_initial(n, seed, first, threads=0, box=b)
    assert r["rc"] == 0
    return r


@pytest.mark.parametrize("model,n", [("glider_v1", 3001), ("glider_v1", 310_003), ("uncor_1200code_v2p1", 5003),
                                     ("terminal_v3_radar_encounter_model", 4001)])
@pytest.mark.parametrize("edge", [B32, B34], ids=["2^32", "2^34"])
def test_initial_across_2_32_and_2_34(model_paths, model, n, edge):
    """k_initial_fast (gather and shared-memory table, fp64 and fp32 values, aligned and unaligned first_sample) across a
    multiple of 2^32 and of 2^34 (there `sample >> 2` changes its high word, so the per-launch call table no longer applies):
    every output byte equals the generic k_initial, and a window around the boundary equals the C oracle.  The terminal
    geometry model is also sampled with its box rejection (generic kernel only), against the C oracle with the same box."""
    import torch
    m = EncounterModel(model_paths[model])
    half = n // 2 // 4 * 4
    for shift in (0, 1, 3):
        first = edge - half - shift
        w0 = half + shift - 500
        ref = _initial_ref(model_paths, model, 1000, 21, first + w0, False)
        for fp32 in (False, True):
            fast = m.sample_initial(n, seed=21, first_sample=first, device="cuda:0", values_fp32=fp32)
            assert L.lib().emb_debug_last_kernel_fast() == 1
            with _generic(1):
                gen = m.sample_initial(n, seed=21, first_sample=first, device="cuda:0", values_fp32=fp32)
                assert L.lib().emb_debug_last_kernel_fast() == 0
            where = "%s first=%d fp32=%d" % (model, first, fp32)
            assert torch.equal(fast[0], gen[0]) and torch.equal(fast[2], gen[2]), where
            if fp32:
                f64 = m.sample_initial(n, seed=21, first_sample=first, device="cuda:0")[1].cpu().numpy()
                for v in (fast[1], gen[1]):
                    assert np.all(np.abs(v.double().cpu().numpy() - f64) <= 1e-6 * np.abs(f64)), where
            else:
                assert torch.equal(fast[1], gen[1]), where
                assert np.array_equal(fast[1].cpu().numpy()[w0:w0 + 1000], ref["values"]), where
            assert np.array_equal(fast[0].cpu().numpy()[w0:w0 + 1000], ref["bins"]), where
            assert np.all(fast[2].cpu().numpy() == 1), where
        if model.startswith("terminal"):
            t = CorTerminalModel(model_paths[model], NARROW, NARROW)
            vals, bins, att = t.sample_raw(n, seed=21, first_sample=first, device="cuda:0")
            assert L.lib().emb_debug_last_kernel_fast() == 0
            rb = _initial_ref(model_paths, model, 1000, 21, first + w0, True)
            where = "terminal box first=%d" % first
            assert int(rb["attempts"].max()) > 1, "the box rejected nothing"
            assert np.array_equal(bins.cpu().numpy()[w0:w0 + 1000], rb["bins"]), where
            assert np.array_equal(vals.cpu().numpy()[w0:w0 + 1000], rb["values"]), where
            assert np.array_equal(att.cpu().numpy()[w0:w0 + 1000].astype(np.int64), rb["attempts"].astype(np.int64)), where


@pytest.mark.parametrize("n_devices", [1, 0], ids=["one", "all"])
def test_multi_device_shard_straddling_2_32(model_paths, n_devices):
    from em_model_manned_bayes_b200.shard import sample_tracks_multi
    m = UncorEncounterModel(model_paths["uncor_1200code_v2p1"])
    n, T, first = 5003, 50, 3 * B32 - 2000
    res, hi, ht = sample_tracks_multi(m, n, T, seed=19, first_sample=first, opts=m.uncor_opts(), n_devices=n_devices)
    hi1 = np.zeros((m.n_initial, 64), dtype=np.uint64)
    ht1 = np.zeros((m.n_dyn, 64), dtype=np.uint64)
    one = m.sample_tracks(n, T, seed=19, first_sample=first, opts=m.uncor_opts(), hist_initial=hi1, hist_transition=ht1)
    assert sum(r.n for r in res) == n
    assert np.array_equal(np.concatenate([r.bins for r in res]), one.bins)
    assert np.array_equal(np.concatenate([r.values for r in res]), one.values)
    assert np.array_equal(np.concatenate([r.init_values for r in res], axis=1), one.init_values)
    assert np.array_equal(np.concatenate([r.attempts for r in res]), one.attempts)
    assert np.array_equal(hi, hi1) and np.array_equal(ht, ht1)
    assert int(ht.sum()) == n * (T - 1) * m.n_dyn


@pytest.fixture(scope="module")
def traj_paths(tmp_path_factory):
    from em_model_manned_bayes_b200.synthetic import write_terminal_model_set
    return write_terminal_model_set(str(tmp_path_factory.mktemp("traj_models")))


def test_terminal_chains_across_2_32_equal_the_emulation(model_paths, traj_paths):
    """create_encounters keyed by encounter indices that straddle a multiple of 2^32: trajectories and chain lengths identical
    to the host emulation"""
    import os
    from em_model_manned_bayes_b200.synthetic import TRAJECTORY_STEMS
    from test_terminal_traj import emu_propagate
    m = CorTerminalModel(model_paths["terminal_v3_radar_encounter_model"])
    m.load_trajectory_models(os.path.dirname(traj_paths[TRAJECTORY_STEMS[0]]))
    vals, _, _ = m.sample_raw(300, seed=4)
    labels = [lab.strip('"') for lab in m.labels_initial]
    geo = np.ascontiguousarray(np.stack([np.asarray(vals)[:, labels.index(f)] for f in CorTerminalModel.GEO_FIELDS]))
    first = 9 * B32 - 77
    res = m.create_encounters(geo, 90, seed=23, first_sample=first, geo_rows=range(12))
    rc, traj, ln = emu_propagate(traj_paths, geo, 23, first, 90)
    assert rc == 0
    assert np.array_equal(np.asarray(res.len), ln)
    assert np.array_equal(np.asarray(res.traj).view(np.uint32), traj.view(np.uint32))


# ---- E. prefix sums over more than 1024 tiles -------------------------------------------------------------------------
def test_event_offsets_past_1024_scan_tiles(model_paths):
    """n = 2^21 + 3 * 2^11 + 5 tracks in one device call: the scan of the tile sums runs its carry over two blocks of 1024.
    Offsets and rows equal two calls below 2^21 tracks joined with their carry; the control rows of expand_events_gpu are
    sized by the same scan and must equal the numpy cumsum of the rows with dt > 0."""
    import torch
    m = UncorEncounterModel(model_paths["uncor_1200code_v2p1"])
    n, T, a = 2 ** 21 + 3 * 2 ** 11 + 5, 6, 2 ** 20 + 7
    ev = m.sample_events(n, T, seed=16, opts=m.uncor_opts(), device="cuda:0")
    parts = [m.sample_events(k, T, seed=16, first_sample=f, opts=m.uncor_opts(), device="cuda:0", want_init=False)
             for f, k in ((0, a), (a, n - a))]
    off = _np(ev.offsets)
    rows = _np(ev.events)
    joff, jrows = _joined([(q.offsets, _np(q.events)) for q in parts])
    assert np.array_equal(off, joff) and np.array_equal(rows, jrows)
    assert off[-1] == ev.total and np.all(np.diff(off) >= 1)
    r = rows.view(L.EVENT_DTYPE)
    assert np.all(r["var"][off[1:] - 1] == 0) and np.count_nonzero(r["var"] == 0) == n
    _, ctl = m.expand_events_gpu(ev, want_samples=False)
    torch.cuda.synchronize()
    per_track = np.add.reduceat((r["dt"] > 0).astype(np.int64), off[:-1])
    assert np.array_equal(_np(ctl.offsets), np.concatenate([[0], np.cumsum(per_track)]))


# ---- F. more than 2^31 rows in one list -------------------------------------------------------------------------------
def test_packed_list_of_more_than_2_31_rows(model_paths):
    """The flagship model, packed rows on the device, T = 1023, enough tracks for about 2.3e9 rows.  The last 10 000 tracks
    equal a separate call for those tracks (rows bit-exact, offsets rebased), and scoring and expanding them from the full
    buffers with their absolute offsets (> 2^31) gives what the separate call's rows give."""
    import torch
    m = UncorEncounterModel(model_paths["uncor_allcode_fwsingle_v1"])
    T, tail = 1023, 10_000
    probe = m.sample_events_packed(200_000, T, seed=17, opts=m.uncor_opts(), device="cuda:0", want_init=False, capacity=1)
    per = probe.total / 200_000
    del probe
    n = int(1.07 * 2 ** 31 / per) + tail
    big = m.sample_events_packed(n, T, seed=17, opts=m.uncor_opts(), device="cuda:0", capacity=1)
    print("\n%d tracks x %d s: %d packed rows (%.1f per track)" % (n, T, big.total, big.total / n))
    assert big.total > 2 ** 31 + 2 ** 26
    off = big.offsets
    a = int(off[n - tail])
    assert a > 2 ** 31
    sep = m.sample_events_packed(tail, T, seed=17, first_sample=n - tail, opts=m.uncor_opts(), device="cuda:0")
    assert torch.equal(off[n - tail:] - a, sep.offsets) and int(off[n]) - a == sep.total
    assert torch.equal(big.words[a:], sep.words) and torch.equal(big.dts[a:], sep.dts)
    for f in ("init_bins", "init_values", "attempts"):
        assert torch.equal(getattr(big, f)[..., n - tail:], getattr(sep, f))
    # the tail tracks read in place from the full buffers: offsets beyond 2^31
    abs_off = off[n - tail:].contiguous()
    ib, iv = big.init_bins[:, n - tail:].contiguous(), big.init_values[:, n - tail:].contiguous()
    got = m.loglik_events(big.words, offsets=abs_off, T=T, init_bins=ib, dts=big.dts)
    want = m.loglik_events(sep)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    _, gc = m.expand_events_gpu(big.words, offsets=abs_off, T=T, init_values=iv, dts=big.dts, want_samples=False,
                                spec=m.out_eme_spec())
    _, wc = m.expand_events_gpu(sep, want_samples=False, spec=m.out_eme_spec())
    torch.cuda.synchronize()
    assert torch.equal(gc.offsets, wc.offsets) and torch.equal(gc.rows, wc.rows)
    del big, got, gc
    torch.cuda.empty_cache()
    L.lib().emb_trim_device_memory(-1)
