"""CPU suite for the em_sample text formatter (emb_format.cuh, emb_format_em_sample): the __host__ __device__ digit generation
and row routines, run on the host by the TEST-ONLY emulation in tests/emu/emu_format.cpp, against Python's '%g' and libc's
snprintf("%g") on edge values and sweeps of millions of doubles, and the row assembly against a Python statement of the rows
em_sample.py writes; the refusals of the C ABI that need no device."""
import ctypes as C
import ctypes.util
import os
import subprocess
import tempfile

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel, tile
from helpers import ROOT

_emu = None


def emu():
    """Build (once per process, into a temporary directory: the tree may be read-only) and load the emulation."""
    global _emu
    if _emu is None:
        out = os.path.join(tempfile.mkdtemp(prefix="emb_format_emu_"), "libemb_format_emu.so")
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared",
                        "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "emu", "emu_format.cpp"), "-o", out],
                       check=True)
        lib = C.CDLL(out)
        vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
        lib.emu_format_g.argtypes = [vp, i64, vp, vp]
        lib.emu_format_em_sample.argtypes = [i64, i32, i64, i32, i32, i32, vp, vp, vp, i32, vp, vp]
        _emu = lib
    return _emu


def emu_g(values):
    """the emulation's "%g" of every value, as a list of str (and the non-finite flag)"""
    v = np.ascontiguousarray(values, dtype=np.float64)
    off = np.zeros(len(v) + 1, dtype=np.int64)
    lib = emu()
    lib.emu_format_g(v.ctypes.data, len(v), None, off.ctypes.data)
    buf = np.zeros(max(1, int(off[-1])), dtype=np.uint8)
    bad = lib.emu_format_g(v.ctypes.data, len(v), buf.ctypes.data, off.ctypes.data)
    b = buf.tobytes()
    return [b[off[i]:off[i + 1]].decode() for i in range(len(v))], bad


def emu_text(n, T, first_id, n_initial, dyn_cols, n_tv, init_values, values_tiled, transition):
    """one text of emb_format_em_sample from the emulation: (bytes, offsets)"""
    cols = np.ascontiguousarray(dyn_cols if len(dyn_cols) else [0], dtype=np.int32)
    iv = np.ascontiguousarray(init_values, dtype=np.float64) if init_values is not None else np.zeros(1)
    vt = np.ascontiguousarray(values_tiled, dtype=np.float32) if values_tiled is not None else np.zeros(1, np.float32)
    off = np.zeros(n + 1, dtype=np.int64)
    lib = emu()
    args = (n, T, first_id, n_initial, len(dyn_cols), n_tv, cols.ctypes.data, iv.ctypes.data, vt.ctypes.data, int(transition))
    st = lib.emu_format_em_sample(*args, None, off.ctypes.data)
    assert st == 0
    buf = np.zeros(max(1, int(off[-1])), dtype=np.uint8)
    assert lib.emu_format_em_sample(*args, buf.ctypes.data, off.ctypes.data) == 0
    return buf.tobytes()[:int(off[-1])], off


_libc = C.CDLL(ctypes.util.find_library("c"))
_libc.snprintf.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_double]


def libc_g(x):
    buf = C.create_string_buffer(64)
    _libc.snprintf(buf, 64, b"%g", float(x))
    return buf.value.decode()


def check_all(values, libc=False):
    values = np.asarray(values, dtype=np.float64)
    got, bad = emu_g(values)
    assert bad == 0
    wrong = [(repr(float(x)), g, "%g" % x) for x, g in zip(values, got) if g != "%g" % x]
    assert not wrong, wrong[:10]
    if libc:
        wrong = [(repr(float(x)), g, libc_g(x)) for x, g in zip(values, got) if g != libc_g(x)]
        assert not wrong, wrong[:10]


EDGES = [(100000.5, "100000"), (100001.5, "100002"), (1234565.0, "1.23456e+06"), (1234575.0, "1.23458e+06"),
         (999999.5, "1e+06"), (999999.4, "999999"), (9.999995e-05, "0.0001"), (1e-05, "1e-05"), (-0.0, "-0"), (0.0, "0"),
         (5e-324, "4.94066e-324"), (1.7976931348623157e308, "1.79769e+308"), (1e100, "1e+100"), (-1.5, "-1.5"),
         (0.0001, "0.0001"), (123456.0, "123456"), (1234567.0, "1.23457e+06")]


@pytest.mark.parametrize("x,want", EDGES)
def test_edge_values(x, want):
    got, _ = emu_g([x])
    assert got[0] == want == "%g" % x == libc_g(x)


def test_powers_of_ten_and_neighbours():
    vals = []
    for k in range(-320, 309):
        p = float("1e%d" % k)
        vals += [p, np.nextafter(p, 0.0), np.nextafter(p, np.inf), -p]
        for d in (999999.5, 999999.4999, 999999.5001, 9999995.0, 100000.5):   # rounding and exponent boundaries at each scale
            q = d * float("1e%d" % (k - 6)) if -300 < k < 300 else p
            vals += [q, np.nextafter(q, 0.0), np.nextafter(q, np.inf)]
    vals += [np.finfo(np.float64).tiny, np.nextafter(np.finfo(np.float64).tiny, 0.0), 5e-324, 1e-323,
             np.finfo(np.float64).max, np.nextafter(np.finfo(np.float64).max, 0.0)]
    check_all(vals, libc=True)


def test_random_bit_patterns():
    rng = np.random.default_rng(20261021)
    v = rng.integers(0, 2 ** 64, size=3_000_000, dtype=np.uint64).view(np.float64)
    check_all(v[np.isfinite(v)])


def test_fp32_widened():
    rng = np.random.default_rng(7)
    f = rng.integers(0, 2 ** 32, size=2_000_000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    f = f[np.isfinite(f)].astype(np.float64)
    # and the magnitudes sampled values take: rates, speeds, altitudes
    g = (rng.standard_normal(1_000_000) * 10.0 ** rng.integers(-3, 6, 1_000_000)).astype(np.float32).astype(np.float64)
    check_all(np.concatenate([f, g]))


def test_exact_ties():
    """(2d+1) 10^k / 2, d of six digits, at every exponent where such a tie is a double: round half to even on the exact value"""
    from fractions import Fraction
    rng = np.random.default_rng(3)
    vals = []
    for k in range(-8, 24):
        f = 5 ** max(-k, 0)                               # for k < 0 the odd numerator must carry 5^-k to be dyadic
        lo, hi = -(-200001 // f), 2000000 // f
        for j in rng.integers(lo, hi, size=12000):
            odd = int(j) * f
            if odd % 2 == 0 or not 200001 <= odd < 2000000:
                continue
            exact = Fraction(odd * 10 ** max(k, 0), 2 * 10 ** max(-k, 0))
            x = float(exact)
            if Fraction(x) == exact:
                vals.append(x)
    assert len(vals) > 100000
    check_all(vals)
    check_all(vals[::10], libc=True)


def test_non_finite_is_flagged():
    for x in (np.inf, -np.inf, np.nan):
        _, bad = emu_g([1.0, x])
        assert bad == 1


def rows_initial(iv, first_id):
    """em_sample.py's initial rows before the device formatter: "%d " % id + " ".join("%g") + "\\n" """
    return "".join("%d " % (first_id + k) + " ".join("%g" % x for x in iv[:, k]) + "\n" for k in range(iv.shape[1]))


def rows_transition(vals, first_id):
    """em_sample.py's transition rows: "%g %g " % (id, t) + " ".join("%g") + "\\n"; vals (n, n_dyn, T) float64"""
    out = []
    for k in range(vals.shape[0]):
        ii = first_id + k
        rows = vals[k].T
        out.append("".join("%g %g " % (ii, j) + " ".join("%g" % x for x in rows[j]) + "\n" for j in range(vals.shape[2])))
    return "".join(out)


@pytest.mark.parametrize("n,T,first_id", [(1, 1, 1), (3, 7, 999_998), (130, 5, 999_900), (260, 60, 1), (5, 3, 2 ** 53 - 5)])
def test_row_assembly(n, T, first_id):
    rng = np.random.default_rng(n * 1000 + T)
    n_initial, n_tv = 16, 6
    dyn_cols = [3, 0, 5, 2]
    iv = rng.standard_normal((n_initial, n)) * 10.0 ** rng.integers(-6, 7, (n_initial, n))
    iv[0, 0] = -0.0
    vals = (rng.standard_normal((n, n_tv, T)) * 10.0 ** rng.integers(-5, 6, (n, n_tv, T))).astype(np.float32)
    text, off = emu_text(n, T, first_id, n_initial, dyn_cols, n_tv, iv, None, False)
    assert text.decode() == rows_initial(iv, first_id)
    assert off[-1] == len(text)
    want = rows_transition(vals[:, dyn_cols, :].astype(np.float64), first_id)
    text, off = emu_text(n, T, first_id, n_initial, dyn_cols, n_tv, None, tile(vals), True)
    assert text.decode() == want
    lines = want.splitlines(keepends=True)
    assert all(text[off[s]:off[s + 1]].decode() == "".join(lines[s * T:(s + 1) * T]) for s in range(n))


# ---- refusals of the C ABI before the device is touched ------------------------------------------------------------------

def _call(m, n, T, first_id, mem=L.EMB_MEM_HOST, transition=True):
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem = mem
    iv = np.zeros((m.n_initial, max(n, 1)))
    off = np.zeros(n + 1, dtype=np.int64)
    vt = np.zeros(1, dtype=np.float32) if transition else None   # every call here is refused before the values are read
    rc = L.lib().emb_format_em_sample(m._h, n, T, first_id, iv.ctypes.data, None if vt is None else vt.ctypes.data, C.byref(o),
                                      0, None, off.ctypes.data, 0, None, off.ctypes.data if transition else None, None)
    return rc, L.lib().emb_last_error().decode()


def test_host_refusals(model_paths):
    m = EncounterModel(model_paths["cor_v1"])
    assert _call(m, 4, 60, 1, mem=L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC)[0] == L.EMB_E_ARG
    assert _call(m, 4, 0, 1)[0] == L.EMB_E_ARG
    assert _call(m, 4, 60, 0)[0] == L.EMB_E_ARG
    rc, msg = _call(m, 4, 60, 2 ** 53 - 3)
    assert rc == L.EMB_E_ARG and "2^53" in msg
    assert _call(m, 1, 2 ** 31 - 1, 1)[0] == L.EMB_E_LIMIT
    t = EncounterModel(model_paths["terminal_v3_radar_encounter_model"])   # no dynamic variables
    rc, msg = _call(t, 4, 60, 1)
    assert rc == L.EMB_E_ARG and "dynvar:empty" in msg
