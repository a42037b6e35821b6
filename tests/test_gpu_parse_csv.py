"""GPU suite for the decimal table parser and the CSV formatter of sample2track (`-m gpu`, on the B200): k_parse_* through
emb_parse_table and k_format_csv[_count] through emb_format_tracks_csv, with host and device buffers, against the host
emulation and Python's float() / '%.0f'; the capacity protocol; a full-size transition.txt body; and the file-to-file driver
sample2track against the host driver it replaced (np.loadtxt, integrate_tracks, the '%' loop), byte for byte over the whole
directory tree."""
import ctypes as C
import math
import os
import random

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from test_parse_csv import bits, csv_rows, emu_csv, emu_parse

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _opts(mem=L.EMB_MEM_HOST):
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem = mem
    return o


def _token_text(seed, count):
    """one text of every kind of token the CPU suite checks, 4 per line"""
    rng = np.random.default_rng(seed)
    f = rng.integers(0, 2 ** 32, size=count, dtype=np.uint64).astype(np.uint32).view(np.float32)
    toks = ["%g" % x for x in f[np.isfinite(f)].astype(np.float64)]
    toks += ["%d" % i for i in rng.integers(1, 2 ** 53, count // 4)] + ["%g" % i for i in rng.integers(1, 2 ** 31, count // 4)]
    r = random.Random(seed)
    for _ in range(count):
        nd = r.randint(1, 19)
        t = "%s%de%d" % (r.choice(("", "-")), r.randrange(10 ** (nd - 1), 10 ** nd), r.randint(-350, 300))
        if abs(float(t)) != float("inf"):
            toks.append(t)
    toks += ["-0", "0e5", ".5", "5.", "+1", "000123.4500", "12345678901234567890000000", "9007199254740993",
             "2.4703282292062328e-324", "1.7976931348623157e308", "4.9406564584124654e-324"]
    toks += ["0"] * ((-len(toks)) % 4)
    lines = [" ".join(toks[i:i + 4]) for i in range(0, len(toks), 4)]
    lines[3] = "\t" + lines[3] + " \r"
    lines.insert(7, "  \r")
    return ("\n".join(lines)).encode(), toks


def test_parse_equals_emulation_and_float_host_and_device():
    from em_model_manned_bayes_b200.sample2track import parse_table
    text, toks = _token_text(3, 400_000)
    rc, want, _, _ = emu_parse(text, 4)
    assert rc == 0
    assert np.array_equal(bits(want.reshape(-1)), bits(np.array([float(t) for t in toks])))
    host = parse_table(text, 4)
    assert isinstance(host, np.ndarray) and np.array_equal(bits(host), bits(want))
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    dev = parse_table(t, 4)
    assert dev.is_cuda and np.array_equal(bits(dev.cpu().numpy()), bits(want))
    # an unaligned device text (the byte path of line discovery) and a text without a final newline
    big = torch.zeros(len(text) + 3, dtype=torch.uint8, device="cuda")
    big[3:] = t
    assert np.array_equal(bits(parse_table(big[3:], 4).cpu().numpy()), bits(want))
    for body in (b"1 2\r\n3 4\r\n", b"\n\n 1 2 \n\r\n \t \n3 4\n\n", b"1\t2\n3 4"):
        for x in (body, torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()):
            assert np.array_equal(_np(parse_table(x, 2)), [[1, 2], [3, 4]])


def test_parse_refusals_and_capacity():
    from em_model_manned_bayes_b200.sample2track import parse_table
    lib = L.lib()
    rows = ["1 2 3"] * 5000
    for tok, kind in (("1e309", "infinity"), ("12345678901234567891", "19"), ("nan", "decimal"), ("1 2", "fields")):
        r = list(rows)
        r[4321] = "4 %s 6" % tok
        for dev in (False, True):
            text = ("\n".join(r) + "\n").encode()
            x = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda() if dev else text
            with pytest.raises(L.EmbError) as ei:
                parse_table(x, 3)
            assert ei.value.code == L.EMB_E_ARG and "line 4322" in str(ei.value) and kind in str(ei.value)
        buf = np.frombuffer(text, dtype=np.uint8).copy()
        got, bad = C.c_int64(), C.c_int64()
        assert lib.emb_parse_table(buf.ctypes.data, len(buf), 3, C.byref(_opts()), 0, None, C.byref(got), C.byref(bad)) == L.EMB_E_ARG
        assert bad.value == 4322
    text = ("\n".join(rows) + "\n\n").encode()
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    vals = torch.full((5000, 3), -7.0, dtype=torch.float64, device="cuda")
    got, bad = C.c_int64(-1), C.c_int64(-1)
    o = _opts(L.EMB_MEM_DEVICE)
    assert lib.emb_parse_table(t.data_ptr(), len(text), 3, C.byref(o), 4999, vals.data_ptr(), C.byref(got), C.byref(bad)) == L.EMB_E_LIMIT
    assert got.value == 5000 and bad.value == 0 and bool((vals == -7.0).all())        # no value written
    assert lib.emb_parse_table(t.data_ptr(), len(text), 3, C.byref(o), 5000, vals.data_ptr(), C.byref(got), C.byref(bad)) == 0
    assert torch.equal(vals, torch.tensor([[1.0, 2.0, 3.0]], device="cuda").expand(5000, 3))


def test_format_csv_equals_emulation_host_and_device():
    from em_model_manned_bayes_b200.sample2track import format_tracks_csv
    rng = np.random.default_rng(9)
    n, T = 1000, 67
    xyz = (rng.standard_normal((3, T + 1, n)) * 10.0 ** rng.integers(-2, 7, (3, T + 1, n))).astype(np.float32)
    xyz[:, 0, ::7] = -0.0
    f = rng.integers(0, 2 ** 32, size=(3, T + 1, 40), dtype=np.uint64).astype(np.uint32).view(np.float32)
    xyz[:, :, -40:] = np.where(np.isfinite(f), f, 1.5)                                   # every magnitude, up to FLT_MAX
    xyz.flat[:6] = [-0.4, 0.5, 1.5, 2.5, -2.5, 2.0 ** 23 + 1]
    mask = (rng.random(n) < 0.8).astype(np.uint8)
    want, want_off = emu_csv(xyz, mask)
    assert want == b"".join(csv_rows(xyz, k) if mask[k] else b"" for k in range(n))
    text, off = format_tracks_csv(xyz, mask)
    assert text.tobytes() == want and np.array_equal(off, want_off)
    text, off = format_tracks_csv(torch.from_numpy(xyz).cuda(), torch.from_numpy(mask).cuda())
    assert text.is_cuda and text.cpu().numpy().tobytes() == want and np.array_equal(off.cpu().numpy(), want_off)
    text, off = format_tracks_csv(xyz)
    assert text.tobytes() == emu_csv(xyz)[0]
    bad = xyz.copy()
    bad[2, T, 5] = np.inf
    m2 = mask.copy()
    m2[5] = 0
    format_tracks_csv(bad, m2)                                                           # masked: not read
    m2[5] = 1
    with pytest.raises(L.EmbError) as ei:
        format_tracks_csv(torch.from_numpy(bad).cuda(), torch.from_numpy(m2).cuda())
    assert ei.value.code == L.EMB_E_ARG and "finite" in str(ei.value)


def test_format_csv_capacity_protocol():
    rng = np.random.default_rng(4)
    n, T = 300, 20
    xyz = torch.from_numpy((rng.standard_normal((3, T + 1, n)) * 1e5).astype(np.float32)).cuda()
    want, want_off = emu_csv(xyz.cpu().numpy())
    lib = L.lib()
    o = _opts(L.EMB_MEM_DEVICE)
    off = torch.full((n + 1,), -1, dtype=torch.int64, device="cuda")
    buf = torch.zeros(len(want) - 1, dtype=torch.uint8, device="cuda")
    total = C.c_int64()
    rc = lib.emb_format_tracks_csv(n, T, xyz.data_ptr(), None, C.byref(o), len(want) - 1, buf.data_ptr(), off.data_ptr(), C.byref(total))
    assert rc == L.EMB_E_LIMIT and total.value == len(want)
    assert np.array_equal(off.cpu().numpy(), want_off) and int(buf.count_nonzero()) == 0
    buf = torch.zeros(len(want), dtype=torch.uint8, device="cuda")
    rc = lib.emb_format_tracks_csv(n, T, xyz.data_ptr(), None, C.byref(o), len(want), buf.data_ptr(), off.data_ptr(), C.byref(total))
    assert rc == 0 and buf.cpu().numpy().tobytes() == want
    rc = lib.emb_format_tracks_csv(n, T, xyz.data_ptr(), None, C.byref(o), 0, None, None, C.byref(total))   # sizing only
    assert rc == L.EMB_E_LIMIT and total.value == len(want)
    for mem, dev in ((L.EMB_MEM_HOST, None), (L.EMB_MEM_DEVICE, "cuda")):
        z = np.full(1, -1, dtype=np.int64) if dev is None else torch.full((1,), -1, dtype=torch.int64, device=dev)
        ptr = z.ctypes.data if dev is None else z.data_ptr()
        assert lib.emb_format_tracks_csv(0, T, None, None, C.byref(_opts(mem)), 0, None, ptr, C.byref(total)) == 0 and int(z[0]) == 0


def test_parse_full_size_transition_text(model_paths):
    """the transition.txt body emb_format_em_sample writes for 1e5 x 600 s of uncor_allcode_fwsingle_v1, parsed on the device"""
    from em_model_manned_bayes_b200.model import EncounterModel
    from em_model_manned_bayes_b200.sample2track import parse_table
    m = EncounterModel(model_paths["uncor_allcode_fwsingle_v1"], idxZeroBoundaries=(1, 2, 3))
    n, T = 100_000, 600
    res = m.sample_tracks(n, T, seed=42, device="cuda", want_bins=False)
    _, _, text, _ = m.format_em_sample(None, res.values_tiled, T, n=n)
    nd = len(m.temporal_map)
    v = parse_table(text, 2 + nd)
    assert v.shape == (n * T, 2 + nd)
    ids = torch.arange(1, n + 1, dtype=torch.float64, device="cuda").repeat_interleave(T)
    assert torch.equal(v[:, 0], torch.where(ids < 1e6, ids, v[:, 0]))                    # ids below 1e6 print exactly
    assert torch.equal(v[:, 1], torch.arange(T, dtype=torch.float64, device="cuda").repeat(n))
    h = text.cpu().numpy()
    starts = np.concatenate([[0], np.flatnonzero(h == 10) + 1])
    pick = np.random.default_rng(1).choice(n * T, 100_000, replace=False)
    got = v[torch.from_numpy(pick).cuda()].cpu().numpy()
    want = np.array([[float(x) for x in h[starts[r]:starts[r + 1]].tobytes().split()] for r in pick])
    assert np.array_equal(bits(got), bits(want))
    # the fp32 values round-trip through "%g" to within its 6 digits
    vals = res.values[:, [list(m.timevarying_vars).index(int(k)) for k in m.temporal_map[:, 0]], :].permute(0, 2, 1).reshape(n * T, nd)
    assert torch.allclose(v[:, 2:], vals.to(torch.float64), rtol=6e-6, atol=0)


# ---- the file-to-file driver ---------------------------------------------------------------------------------------------------

def host_sample2track(parameters_filename, initial_filename, transition_filename, num_max_tracks=10000, out_dir_parent="out",
                      rng_seed=42):
    """sample2track.py before the device parser and formatter: np.loadtxt, integrate_tracks on host buffers, the '%' loop"""
    from em_model_manned_bayes_b200.model import EncounterModel, TrackResult, tile
    from em_model_manned_bayes_b200.sample2track import _find, integrate_opts, integrate_tracks, make_valid_name

    def read(path):
        with open(path, encoding="utf-8") as f:
            f.readline()
            return np.loadtxt(f, ndmin=2)

    model = EncounterModel(parameters_filename, idxZeroBoundaries=(1, 2, 3), isOverwriteZeroBoundaries=False)
    o = integrate_opts(model)
    names_init = [make_valid_name(l) for l in model.labels_initial]
    dyn_t = [int(v) for v in model.temporal_map[:, 0]]
    Ti, Tt = read(initial_filename), read(transition_filename)
    if Ti.shape[0] > num_max_tracks:
        keep = np.sort(np.random.default_rng(rng_seed).permutation(Ti.shape[0])[:num_max_tracks])
        Ti = Ti[keep]
    n = Ti.shape[0]
    ids = Ti[:, 0].astype(np.int64)
    Tt = Tt[np.argsort(Tt[:, 0], kind="stable")]
    first = np.searchsorted(Tt[:, 0], ids, side="left")
    last = np.searchsorted(Tt[:, 0], ids, side="right")
    T = int(last[0] - first[0])
    if T < 1 or np.any(last - first != T):
        raise L.EmbError(L.EMB_E_ARG, "sample2track: every track needs the same number of transition rows")
    rows = (first[:, None] + np.arange(T)[None, :]).ravel()
    upd = Tt[rows, 2:].reshape(n, T, len(dyn_t))
    tv = list(model.timevarying_vars)
    dense = np.zeros((n, len(tv), T), dtype=np.float32)
    for k, v in enumerate(dyn_t):
        dense[:, tv.index(v), :] = upd[:, :, k]
    res = TrackResult(n=n, T=T, dyn_vars=dyn_t, tv_vars=tv, bins_tiled=None, values_tiled=tile(dense), init_bins=None,
                      init_values=np.ascontiguousarray(Ti[:, 1:].T), attempts=None)
    xyz, good = integrate_tracks(model, res, opts=o)
    is_good = good.astype(bool)
    b_alt = model.boundaries[o.idx_altitude - 1]
    min_alt, max_alt = float(b_alt[0]), float(b_alt[-1])
    Ls = np.arange(math.floor(min_alt - 50) if min_alt % 100 else min_alt, max_alt + 200 + 1e-9, 100.0)
    if Ls[0] < 0:
        Ls[0] = 0
    iG, iA = _find(names_init, "G"), _find(names_init, "A")
    speed0 = Ti[:, o.idx_speed] * o.ur_speed
    for k in np.nonzero(is_good)[0]:
        z0 = float(xyz[2, 0, k])
        parts = []
        if iG:
            parts.append("G%d" % int(Ti[k, iG]))
        if iA:
            parts.append("A%d" % int(Ti[k, iA]))
        j = int(np.searchsorted(Ls, z0, side="right")) - 1
        parts.append("%dft" % int(Ls[min(max(j, 0), len(Ls) - 2)]))
        d = os.path.join(out_dir_parent, *parts)
        os.makedirs(d, exist_ok=True)
        name = "BAYES_t%d_id%d_alt%d_speed%d.csv" % (T, k + 1, int(math.floor(z0 + 0.5)), int(math.floor(speed0[k] + 0.5)))
        with open(os.path.join(d, name), "w", encoding="utf-8") as f:
            f.write("time_s,x_ft,y_ft,z_ft\n")
            f.write("".join("%d,%.0f,%.0f,%.0f\n" % (t, xyz[0, t, k], xyz[1, t, k], xyz[2, t, k]) for t in range(T + 1)))
    Tc = Ti.copy()
    Tc[:, o.idx_speed] *= o.ur_speed
    Tc[:, o.idx_acceleration] *= o.ur_speed
    Tc[:, o.idx_vertrate] *= o.ur_vertrate
    return is_good, Tc


def tree(root):
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            p = os.path.join(d, f)
            out[os.path.relpath(p, root)] = open(p, "rb").read()
    return out


@pytest.mark.parametrize("model,n,T,max_tracks,crlf", [("uncor_1200code_v2p1", 3000, 120, 10000, False),
                                                       ("uncor_1200code_v2p1", 3000, 120, 1000, True),
                                                       ("uncor_allcode_fwsingle_v1", 2000, 601, 10000, True),
                                                       ("uncor_allcode_fwsingle_v1", 2000, 301, 777, False)])
def test_sample2track_tree_equals_host_driver(model_paths, tmp_path, model, n, T, max_tracks, crlf):
    from em_model_manned_bayes_b200.em_sample import em_sample
    from em_model_manned_bayes_b200.sample2track import sample2track
    fi, ft = str(tmp_path / "initial.txt"), str(tmp_path / "transition.txt")
    em_sample(model_paths[model], fi, ft, num_initial_samples=n, num_transition_samples=T, rng_seed=7)
    if crlf:
        for p in (fi, ft):
            data = open(p, "rb").read().replace(b"\n", b"\r\n")
            open(p, "wb").write(data)
    want_good, want_tc = host_sample2track(model_paths[model], fi, ft, num_max_tracks=max_tracks, out_dir_parent=str(tmp_path / "host"))
    got_good, got_tc = sample2track(model_paths[model], fi, ft, num_max_tracks=max_tracks, out_dir_parent=str(tmp_path / "dev"))
    assert np.array_equal(got_good, want_good) and got_good.dtype == want_good.dtype
    assert np.array_equal(bits(got_tc), bits(want_tc))
    a, b = tree(str(tmp_path / "host")), tree(str(tmp_path / "dev"))
    assert len(a) == int(want_good.sum()) > 0
    assert sorted(a) == sorted(b)
    assert all(a[k] == b[k] for k in a)


def test_sample2track_refuses_like_the_host_driver(model_paths, tmp_path):
    """ids from 1,000,000 on print as %g in transition.txt and collide: both drivers fail with the equal-T error"""
    from em_model_manned_bayes_b200.sample2track import sample2track
    m = "uncor_1200code_v2p1"
    from em_model_manned_bayes_b200.model import EncounterModel
    mdl = EncounterModel(model_paths[m], idxZeroBoundaries=(1, 2, 3))
    n, T = 4, 3
    res = mdl.sample_tracks(n, T, seed=1)
    ti, _, tt, _ = mdl.format_em_sample(res, first_id=999_998)
    fi, ft = str(tmp_path / "i.txt"), str(tmp_path / "t.txt")
    open(fi, "wb").write(b"id x\n" + ti.tobytes())
    open(ft, "wb").write(b"initial_id t x\n" + tt.tobytes())
    for fn in (host_sample2track, sample2track):
        with pytest.raises(L.EmbError) as ei:
            fn(model_paths[m], fi, ft, out_dir_parent=str(tmp_path / "o"))
        assert "same number of transition rows" in str(ei.value)
