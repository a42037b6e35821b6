"""CPU suite for the decimal table parser (emb_parse.cuh, emb_parse_table) and the CSV formatter of sample2track (emb_format.cuh:
format_csv_track, emb_format_tracks_csv): the __host__ __device__ per-line and per-track routines, run on the host by the
TEST-ONLY emulation in tests/emu/emu_parse_csv.cpp, against Python's float() bit for bit and Python's '%.0f' byte for byte;
the refusals of the C ABI that need no device."""
import ctypes as C
import os
import random
import struct
import subprocess
import tempfile
from fractions import Fraction

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from helpers import ROOT

_emu = None

E_TOKEN, E_DIGITS, E_RANGE, E_FIELDS = 0, 1, 2, 3


def emu():
    """Build (once per process, into a temporary directory: the tree may be read-only) and load the emulation."""
    global _emu
    if _emu is None:
        out = os.path.join(tempfile.mkdtemp(prefix="emb_parse_emu_"), "libemb_parse_emu.so")
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared",
                        "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "emu", "emu_parse_csv.cpp"), "-o", out],
                       check=True)
        lib = C.CDLL(out)
        vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
        lib.emu_parse_table.argtypes = [vp, i64, i32, i64, vp, vp, vp, vp]
        lib.emu_format_f0.argtypes = [vp, i64, vp, vp]
        lib.emu_format_tracks_csv.argtypes = [i64, i32, vp, vp, vp, vp]
        _emu = lib
    return _emu


def emu_parse(text: bytes, cols: int, capacity=None):
    """-> (rc, values (rows, cols), bad_line, kind) of the emulation"""
    buf = np.frombuffer(text, dtype=np.uint8).copy() if text else np.zeros(1, np.uint8)
    cap = (len(text) + 1) // (2 * cols) if capacity is None else capacity
    vals = np.zeros(max(cap, 1) * cols)
    tot, bad, kind = C.c_int64(), C.c_int64(), C.c_int32()
    rc = emu().emu_parse_table(buf.ctypes.data, len(text), cols, cap, vals.ctypes.data, C.byref(tot), C.byref(bad), C.byref(kind))
    return rc, vals[:tot.value * cols].reshape(-1, cols), bad.value, kind.value


def emu_f0(values):
    """the emulation's "%.0f" of every float32, as a list of str (and the non-finite flag)"""
    v = np.ascontiguousarray(values, dtype=np.float32)
    off = np.zeros(len(v) + 1, dtype=np.int64)
    lib = emu()
    lib.emu_format_f0(v.ctypes.data, len(v), None, off.ctypes.data)
    buf = np.zeros(max(1, int(off[-1])), dtype=np.uint8)
    bad = lib.emu_format_f0(v.ctypes.data, len(v), buf.ctypes.data, off.ctypes.data)
    b = buf.tobytes()
    return [b[off[i]:off[i + 1]].decode() for i in range(len(v))], bad


def emu_csv(xyz, mask=None):
    """emb_format_tracks_csv from the emulation: (bytes, offsets)"""
    x = np.ascontiguousarray(xyz, dtype=np.float32)
    T, n = x.shape[1] - 1, x.shape[2]
    mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
    off = np.zeros(n + 1, dtype=np.int64)
    lib = emu()
    args = (n, T, x.ctypes.data, None if mk is None else mk.ctypes.data)
    assert lib.emu_format_tracks_csv(*args, None, off.ctypes.data) == 0
    buf = np.zeros(max(1, int(off[-1])), dtype=np.uint8)
    assert lib.emu_format_tracks_csv(*args, buf.ctypes.data, off.ctypes.data) == 0
    return buf.tobytes()[:int(off[-1])], off


def csv_rows(xyz, k):
    """the rows sample2track.py wrote for track k before the device formatter"""
    return "".join("%d,%.0f,%.0f,%.0f\n" % (t, xyz[0, t, k], xyz[1, t, k], xyz[2, t, k]) for t in range(xyz.shape[1])).encode()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def check_tokens(tokens, cols=1):
    """every token parsed by the emulation equals float(token) bit for bit (one token per field, `cols` per line)"""
    want = np.array([float(t) for t in tokens])
    pad = (-len(tokens)) % cols
    toks = list(tokens) + ["0"] * pad
    lines = [" ".join(toks[i:i + cols]) for i in range(0, len(toks), cols)]
    rc, v, bad, kind = emu_parse(("\n".join(lines) + "\n").encode(), cols)
    assert rc == 0, (bad, kind, lines[bad - 1] if bad else None)
    got = v.reshape(-1)[:len(tokens)]
    wrong = np.nonzero(bits(got) != bits(want))[0]
    assert not len(wrong), [(tokens[i], repr(got[i]), repr(want[i])) for i in wrong[:10]]


# ---- "%.0f" ---------------------------------------------------------------------------------------------------------------------

def check_f0(values):
    values = np.asarray(values, dtype=np.float32)
    got, bad = emu_f0(values)
    assert bad == 0
    wrong = [(repr(float(x)), g, "%.0f" % float(x)) for x, g in zip(values, got) if g != "%.0f" % float(x)]
    assert not wrong, wrong[:10]


def test_f0_edge_values():
    vals = [0.0, -0.0, 0.4, -0.4, 0.5, -0.5, 1.5, -1.5, 2.5, -2.5, 2.0 ** 23 - 1, 2.0 ** 23 + 1, -(2.0 ** 23 + 1), 2.0 ** 24,
            np.finfo(np.float32).max, -np.finfo(np.float32).max, np.float32(1e-45), -np.float32(1e-45), np.finfo(np.float32).tiny,
            2.0 ** 23 - 0.5, 2.0 ** 22 + 0.5, 0.49999997, 1e10, 2.0 ** 127, 2.0 ** 64 + 2.0 ** 41]
    check_f0(vals)
    got, _ = emu_f0([-0.4, -0.0, 0.5, 1.5, 2.5])
    assert got == ["-0", "-0", "0", "2", "2"]


def test_f0_ties():
    rng = np.random.default_rng(11)
    k = rng.integers(-2 ** 23, 2 ** 23, size=400_000)
    v = (k.astype(np.float64) + 0.5).astype(np.float32)
    assert np.array_equal(v.astype(np.float64), k + 0.5)   # every k + 0.5 with |k| < 2^23 is a float
    check_f0(np.concatenate([v, np.arange(-1000, 1000) + np.float32(0.5)]))


def test_f0_random_bit_patterns():
    rng = np.random.default_rng(20261022)
    f = rng.integers(0, 2 ** 32, size=3_000_000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    check_f0(f[np.isfinite(f)])


def test_f0_non_finite_is_flagged():
    for x in (np.inf, -np.inf, np.nan):
        _, bad = emu_f0([1.0, x])
        assert bad == 1


@pytest.mark.parametrize("n,T", [(1, 0), (7, 1), (33, 60), (130, 31)])
def test_csv_tracks_with_mask(n, T):
    rng = np.random.default_rng(n * 100 + T)
    xyz = (rng.standard_normal((3, T + 1, n)) * 10.0 ** rng.integers(-2, 7, (3, T + 1, n))).astype(np.float32)
    xyz[:, 0, :] = np.where(rng.random((3, n)) < 0.3, -0.0, xyz[:, 0, :])
    xyz.flat[:4] = [-0.4, 0.5, 2.5, np.finfo(np.float32).max][:xyz.size]
    mask = (rng.random(n) < 0.7).astype(np.uint8)
    mask[0] = 1
    for mk in (mask, None):
        text, off = emu_csv(xyz, mk)
        want = b"".join(csv_rows(xyz, k) if mk is None or mk[k] else b"" for k in range(n))
        assert text == want
        for k in range(n):
            assert text[off[k]:off[k + 1]] == (csv_rows(xyz, k) if mk is None or mk[k] else b"")
    bad = xyz.copy()
    bad[1, T, n - 1] = np.nan
    mk = np.ones(n, np.uint8)
    mk[n - 1] = 0
    emu_csv(bad, mk)                                  # a masked track is not read
    off = np.zeros(n + 1, dtype=np.int64)
    assert emu().emu_format_tracks_csv(n, T, bad.ctypes.data, None, None, off.ctypes.data) == 1


# ---- the parser -----------------------------------------------------------------------------------------------------------------

def test_parse_special_tokens():
    toks = ["-0", "0e5", ".5", "5.", "+1", "000123.4500", "-000.000", "0.0e-999999999999", "1e-400", "-1e-400", "1E5", "1e+5",
            "12345678901234567890000000", "0.00000000000000000000012345678901234567890", "1234567890123456789",
            "9007199254740993", "1e22", "1e23", "1e-22", "1e-23", "4.9406564584124654e-324", "2.4703282292062328e-324",
            "2.4703282292062327e-324", "-2.4703282292062328e-324", "2.2250738585072011e-308", "2.2250738585072014e-308",
            "1.7976931348623157e308", "1.7976931348623158e308", "-1.7976931348623158e+308", "17976931348623157e292"]
    check_tokens(toks)
    rc, v, _, _ = emu_parse(b"-0\n0e5\n-0.0e-5\n", 1)
    assert rc == 0 and [struct.pack("<d", x) for x in v[:, 0]] == [struct.pack("<d", x) for x in (-0.0, 0.0, -0.0)]


def test_parse_g_of_fp32_and_ids():
    """every token em_sample writes: "%g" of fp32 values widened to double, ids as "%d" and "%g" """
    rng = np.random.default_rng(5)
    f = rng.integers(0, 2 ** 32, size=3_000_000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    f = f[np.isfinite(f)].astype(np.float64)
    g = (rng.standard_normal(300_000) * 10.0 ** rng.integers(-3, 6, 300_000)).astype(np.float32).astype(np.float64)
    toks = ["%g" % x for x in np.concatenate([f, g])]
    ids = np.concatenate([np.arange(1, 200_001), rng.integers(1, 2 ** 53, 100_000)])
    toks += ["%d" % i for i in ids] + ["%g" % i for i in ids]
    check_tokens(toks, cols=8)


def test_parse_random_mantissas_and_exponents():
    rng = random.Random(19)
    toks = []
    while len(toks) < 600_000:
        nd = rng.randint(1, 19)
        w = rng.randrange(10 ** (nd - 1), 10 ** nd)
        q = rng.randint(-350, 310)
        t = "%s%de%d" % (rng.choice(("", "-")), w, q)
        if nd + q <= 308 or abs(float(t)) != float("inf"):
            toks.append(t)
        if rng.random() < 0.2:   # the same digits with a point inside
            s = str(w)
            k = rng.randint(0, len(s))
            t2 = s[:k] + "." + s[k:] + "e%d" % (q + len(s) - k)
            if abs(float(t2)) != float("inf"):
                toks.append(t2)
    check_tokens(toks, cols=4)


def _halfway(a):
    """the exact halfway point between the positive double a and its successor, as a Fraction"""
    return (Fraction(a) + Fraction(float(np.nextafter(a, np.inf)))) / 2


def _sig19(fr, up, approx):
    """the 19-significant-digit decimal just below (or above, `up`) the positive Fraction fr (about `approx`), as a token"""
    import math
    e = math.floor(math.log10(approx)) - 18
    while fr < Fraction(10) ** (e + 18):
        e -= 1
    while fr >= Fraction(10) ** (e + 19):
        e += 1
    s = fr / Fraction(10) ** e
    d = s.numerator // s.denominator + (1 if up else -1 if s.denominator == 1 else 0)   # strictly below or above
    return "%de%d" % (d, e)


def test_parse_around_halfway_points():
    """Halfway points between adjacent doubles: exactly, where one has at most 19 significant digits (ties to even), and
    across the normal range, the subnormals and up to DBL_MAX as the 19-digit decimals just below and just above it (the
    closest a 19-digit token gets to the tie: it must round down, respectively up)."""
    rng = np.random.default_rng(23)
    ties, near, want_near = [], [], []
    for _ in range(30_000):   # exact ties m 2^j (m odd, 2^53 < m < 2^54) with at most 19 significant digits
        m = int(rng.integers(2 ** 52, 2 ** 53)) * 2 + 1
        j = int(rng.integers(-3, 12))
        fr = Fraction(m) * Fraction(2) ** j
        if fr.denominator == 1:
            s = str(fr.numerator).rstrip("0")
            z = len(str(fr.numerator)) - len(s)
            tok = "%se%d" % (s, z)
        else:
            tok = str(Fraction(fr.numerator * 10 ** 3, fr.denominator).numerator) + "e-3"
        if len(tok.split("e")[0].strip("0")) <= 19:
            ties.append(tok)
    assert len(ties) > 10_000
    check_tokens(ties)
    ex = np.concatenate([rng.integers(-1074, 972, 40_000), np.arange(-1074, -1020), np.arange(960, 972)])
    for e2 in ex:
        a = float(np.ldexp(1.0 + float(rng.random()), int(e2))) if e2 >= -1022 else float(np.ldexp(float(rng.integers(1, 2 ** 52)), -1074))
        if a >= np.finfo(np.float64).max:
            a = float(np.nextafter(np.finfo(np.float64).max, 0))
        h = _halfway(a)
        for up in (False, True):
            near.append(_sig19(h, up, a))
            want_near.append(float(np.nextafter(a, np.inf)) if up else a)
    a = float(np.nextafter(np.finfo(np.float64).max, 0))
    near += [_sig19(_halfway(a), True, a)]
    want_near += [np.finfo(np.float64).max]
    check_tokens(near)
    assert np.array_equal(bits(np.array([float(t) for t in near])), bits(np.array(want_near)))


@pytest.mark.parametrize("tok,kind", [("12345678901234567891", E_DIGITS), ("1.2345678901234567891", E_DIGITS),
                                      ("0.000123456789012345678912", E_DIGITS), ("1e309", E_RANGE), ("-1.8e308", E_RANGE),
                                      ("1.7976931348623159e308", E_RANGE), ("inf", E_TOKEN), ("-inf", E_TOKEN), ("nan", E_TOKEN),
                                      ("0x1p3", E_TOKEN), ("1,5", E_TOKEN), ("1e", E_TOKEN), ("1e+", E_TOKEN), ("--1", E_TOKEN),
                                      ("1..2", E_TOKEN), (".", E_TOKEN), ("+", E_TOKEN), ("e5", E_TOKEN), ("1e5.0", E_TOKEN),
                                      ("1_000", E_TOKEN), ("\x0b1", E_TOKEN)])
def test_parse_refusals_name_the_line(tok, kind):
    for line in (1, 2, 7):
        rows = ["1 2 3"] * 9
        rows[line - 1] = "4 %s 6" % tok
        rc, _, bad, k = emu_parse(("\n".join(rows) + "\n").encode(), 3)
        assert (rc, bad, k) == (-4, line, kind)


def test_parse_field_counts_and_first_error():
    rc, _, bad, k = emu_parse(b"1 2 3\n\n1 2\n", 3)
    assert (rc, bad, k) == (-4, 3, E_FIELDS)
    rc, _, bad, k = emu_parse(b"1 2 3\n1 2 3 4\n", 3)
    assert (rc, bad, k) == (-4, 2, E_FIELDS)
    rc, _, bad, k = emu_parse(b"1 2 3\n1 2 3\n1 x 3\n1 1e999 3\n", 3)   # the first line with an error
    assert (rc, bad, k) == (-4, 3, E_TOKEN)
    rc, _, bad, k = emu_parse(b"1 2 3\n1 1e999 3\n1 x 3\n", 3)
    assert (rc, bad, k) == (-4, 2, E_RANGE)


@pytest.mark.parametrize("body", [b"1 2\n3 4\n", b"1 2\r\n3 4\r\n", b"1\t2\n3\t\t4", b"\n\n 1 2 \n\r\n \t \n3 4\n\n",
                                  b"1 2\r\n\r\n3 4", b"  1   2\n3 4\n   "])
def test_parse_layouts(body):
    rc, v, _, _ = emu_parse(body, 2)
    assert rc == 0 and np.array_equal(v, [[1, 2], [3, 4]])
    import io
    assert np.array_equal(v, np.loadtxt(io.StringIO(body.decode()), ndmin=2))


def test_parse_capacity_and_empty():
    rc, v, _, _ = emu_parse(b"", 3)
    assert rc == 0 and v.shape == (0, 3)
    rc, v, _, _ = emu_parse(b"\n \n\r\n", 3)
    assert rc == 0 and v.shape == (0, 3)
    buf = np.frombuffer(b"1\n2\n3\n", dtype=np.uint8).copy()
    tot, bad, kind = C.c_int64(), C.c_int64(), C.c_int32()
    rc = emu().emu_parse_table(buf.ctypes.data, 6, 1, 2, None, C.byref(tot), C.byref(bad), C.byref(kind))
    assert rc == L.EMB_E_LIMIT and tot.value == 3


# ---- refusals of the C ABI before the device is touched --------------------------------------------------------------------

def _opts(mem=L.EMB_MEM_HOST):
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem = mem
    return o


def test_host_refusals():
    lib = L.lib()
    text = np.frombuffer(b"1 2\n", dtype=np.uint8).copy()
    vals = np.zeros(8)
    rows, bad = C.c_int64(-1), C.c_int64(-1)
    for cols in (0, -1, 257):
        assert lib.emb_parse_table(text.ctypes.data, 4, cols, C.byref(_opts()), 4, vals.ctypes.data, C.byref(rows), C.byref(bad)) == L.EMB_E_ARG
    assert lib.emb_parse_table(text.ctypes.data, -1, 2, C.byref(_opts()), 4, vals.ctypes.data, C.byref(rows), C.byref(bad)) == L.EMB_E_ARG
    rc = lib.emb_parse_table(text.ctypes.data, 4, 2, C.byref(_opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)), 4, vals.ctypes.data,
                             C.byref(rows), C.byref(bad))
    assert rc == L.EMB_E_ARG and "EMB_MEM_ASYNC" in lib.emb_last_error().decode()
    assert lib.emb_parse_table(None, 0, 2, C.byref(_opts()), 0, None, C.byref(rows), C.byref(bad)) == 0 and rows.value == 0
    xyz = np.zeros((3, 2, 1), dtype=np.float32)
    off = np.zeros(2, dtype=np.int64)
    assert lib.emb_format_tracks_csv(1, -1, xyz.ctypes.data, None, C.byref(_opts()), 0, None, off.ctypes.data, None) == L.EMB_E_ARG
    assert lib.emb_format_tracks_csv(-1, 1, xyz.ctypes.data, None, C.byref(_opts()), 0, None, off.ctypes.data, None) == L.EMB_E_ARG
    assert lib.emb_format_tracks_csv(1, 2 ** 31 - 1, xyz.ctypes.data, None, C.byref(_opts()), 0, None, off.ctypes.data,
                                     None) == L.EMB_E_LIMIT
    rc = lib.emb_format_tracks_csv(1, 1, xyz.ctypes.data, None, C.byref(_opts(L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)), 0, None,
                                   off.ctypes.data, None)
    assert rc == L.EMB_E_ARG and "EMB_MEM_ASYNC" in lib.emb_last_error().decode()
    off[:] = -1
    assert lib.emb_format_tracks_csv(0, 5, None, None, C.byref(_opts()), 0, None, off.ctypes.data, None) == 0 and off[0] == 0


def test_tile_torch_equals_numpy():
    torch = pytest.importorskip("torch")
    from em_model_manned_bayes_b200.model import tile, untile
    rng = np.random.default_rng(2)
    for n, nv, T in ((1, 1, 1), (129, 3, 7), (300, 5, 600)):
        v = rng.standard_normal((n, nv, T)).astype(np.float32)
        t = tile(torch.from_numpy(v))
        assert isinstance(t, torch.Tensor) and np.array_equal(t.numpy(), tile(v))
        assert np.array_equal(untile(t, nv, n, T).numpy(), v)
