"""Times of the sample2track text path on the device: the decimal table parser (emb_parse_table), the CSV formatter
(emb_format_tracks_csv) and the file-to-file driver sample2track.

    python tools/time_sample2track.py [OUT_DIR]        (default profiles/)

Workloads (uncor_allcode_fwsingle_v1):
  - emb_parse_table of the transition.txt body emb_format_em_sample writes for 1e5 tracks x 600 s, text and values
    device-resident, capacity known: the whole call (CUDA events, median of 10 after a warm-up), the parse_table helper (sizing
    call included), and the kernels split per kernel (torch.profiler with CUDA activities over 10 more calls, in a separate
    window; per-call medians);
  - emb_format_tracks_csv of emb_tracks_integrate's output for the same 1e5 x 600 s tracks, device-resident, capacity known: the
    same three measurements;
  - sample2track at n = 1e4, T = 600 on files em_sample wrote to local disk, wall clock split into read, parse, integrate
    (grouping by id, tiles and emb_tracks_integrate), format and file writes, against the host driver it replaced (np.loadtxt,
    integrate_tracks on host buffers, the '%' loop; kept below as the comparison) on the same files and disk; and both whole
    calls, whose directory trees must be identical.
Writes sample2track_b200.json into OUT_DIR with the card name, power limit and max SM clock read in the same run (nvidia-smi's
read-only query).
"""
import ctypes as C
import json
import math
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from em_model_manned_bayes_b200 import _lib as L  # noqa: E402
from em_model_manned_bayes_b200 import sample2track as S  # noqa: E402
from em_model_manned_bayes_b200.em_sample import em_sample  # noqa: E402
from em_model_manned_bayes_b200.model import EncounterModel, TrackResult, tile  # noqa: E402
from em_model_manned_bayes_b200.model_archive import materialize  # noqa: E402

MODEL, N, T = "uncor_allcode_fwsingle_v1", 100_000, 600
N_FILES = 10_000


def timed(fn, reps=10, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return {"median": times[len(times) // 2], "min": times[0]}


def kernel_split(fn, pattern, reps=10):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and re.search(pattern, e.name):
            name = re.search(pattern, e.name).group(0)
            kern.setdefault(name, []).append(e.device_time if hasattr(e, "device_time") else e.cuda_time)
    # us -> ms per call (a kernel launched k times per call, like k_scan_*, is summed over its launches)
    return {k: float(np.median(v)) / 1000.0 * (len(v) // reps) for k, v in kern.items()}


def _opts():
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem, o.device, o.stream = L.EMB_MEM_DEVICE, torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream
    return o


def names_and_files(model, o, Ti, xyz_z0, is_good, T, out_dir, rows_of):
    """the directory tree and file names of sample2track (:143-178, :246-290); rows_of(k) -> the bytes of track k"""
    names_init = [S.make_valid_name(l) for l in model.labels_initial]
    b_alt = model.boundaries[o.idx_altitude - 1]
    min_alt, max_alt = float(b_alt[0]), float(b_alt[-1])
    Ls = np.arange(math.floor(min_alt - 50) if min_alt % 100 else min_alt, max_alt + 200 + 1e-9, 100.0)
    if Ls[0] < 0:
        Ls[0] = 0
    iG, iA = S._find(names_init, "G"), S._find(names_init, "A")
    speed0 = Ti[:, o.idx_speed] * o.ur_speed
    for k in np.nonzero(is_good)[0]:
        z0 = float(xyz_z0[k])
        parts = []
        if iG:
            parts.append("G%d" % int(Ti[k, iG]))
        if iA:
            parts.append("A%d" % int(Ti[k, iA]))
        j = int(np.searchsorted(Ls, z0, side="right")) - 1
        parts.append("%dft" % int(Ls[min(max(j, 0), len(Ls) - 2)]))
        d = os.path.join(out_dir, *parts)
        os.makedirs(d, exist_ok=True)
        name = "BAYES_t%d_id%d_alt%d_speed%d.csv" % (T, k + 1, int(math.floor(z0 + 0.5)), int(math.floor(speed0[k] + 0.5)))
        with open(os.path.join(d, name), "wb") as f:
            f.write(b"time_s,x_ft,y_ft,z_ft\n")
            f.write(rows_of(k))


def host_driver_split(path, fi, ft, out_dir):
    """sample2track.py before the device parser and formatter, stage by stage (the comparison)"""
    import io
    t = {}
    t0 = time.perf_counter()
    texts = []
    for p in (fi, ft):
        with open(p, encoding="utf-8") as f:
            f.readline()
            texts.append(f.read())
    t["read_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    Ti, Tt = (np.loadtxt(io.StringIO(x), ndmin=2) for x in texts)
    t["parse_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    model = EncounterModel(path, idxZeroBoundaries=(1, 2, 3))
    o = S.integrate_opts(model)
    dyn_t = [int(v) for v in model.temporal_map[:, 0]]
    n = Ti.shape[0]
    ids = Ti[:, 0].astype(np.int64)
    Tt = Tt[np.argsort(Tt[:, 0], kind="stable")]
    first = np.searchsorted(Tt[:, 0], ids, side="left")
    T_ = int(np.searchsorted(Tt[:, 0], ids[:1], side="right")[0] - first[0])
    upd = Tt[(first[:, None] + np.arange(T_)[None, :]).ravel(), 2:].reshape(n, T_, len(dyn_t))
    tv = list(model.timevarying_vars)
    dense = np.zeros((n, len(tv), T_), dtype=np.float32)
    for k, v in enumerate(dyn_t):
        dense[:, tv.index(v), :] = upd[:, :, k]
    res = TrackResult(n=n, T=T_, dyn_vars=dyn_t, tv_vars=tv, bins_tiled=None, values_tiled=tile(dense), init_bins=None,
                      init_values=np.ascontiguousarray(Ti[:, 1:].T), attempts=None)
    xyz, good = S.integrate_tracks(model, res, opts=o)
    t["integrate_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    is_good = good.astype(bool)
    rows = {int(k): "".join("%d,%.0f,%.0f,%.0f\n" % (s, xyz[0, s, k], xyz[1, s, k], xyz[2, s, k]) for s in range(T_ + 1)).encode()
            for k in np.nonzero(is_good)[0]}
    t["format_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    names_and_files(model, o, Ti, xyz[2, 0], is_good, T_, out_dir, lambda k: rows[int(k)])
    t["write_s"] = time.perf_counter() - t0
    return t


def device_driver_split(path, fi, ft, out_dir):
    """sample2track's device path stage by stage, each stage ending in a synchronise"""
    t = {}
    dev = torch.device("cuda", torch.cuda.current_device())
    t0 = time.perf_counter()
    bi, bt = S._to_device(fi, dev), S._to_device(ft, dev)
    torch.cuda.synchronize()
    t["read_s"] = time.perf_counter() - t0
    model = EncounterModel(path, idxZeroBoundaries=(1, 2, 3))
    o = S.integrate_opts(model)
    dyn_t = [int(v) for v in model.temporal_map[:, 0]]
    t0 = time.perf_counter()
    Ti = S.parse_table(bi, 1 + model.n_initial)
    Tt = S.parse_table(bt, 2 + len(dyn_t))
    torch.cuda.synchronize()
    t["parse_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    n = int(Ti.shape[0])
    ids = Ti[:, 0].to(torch.int64).to(torch.float64)
    key, order = torch.sort(Tt[:, 0], stable=True)
    Tt = Tt[order]
    first = torch.searchsorted(key, ids, side="left")
    cnt = (torch.searchsorted(key, ids, side="right") - first).cpu().numpy()
    T_ = int(cnt[0])
    upd = Tt[(first[:, None] + torch.arange(T_, device=dev)[None, :]).reshape(-1), 2:].reshape(n, T_, len(dyn_t))
    tv = list(model.timevarying_vars)
    dense = torch.zeros((n, len(tv), T_), dtype=torch.float32, device=dev)
    for k, v in enumerate(dyn_t):
        dense[:, tv.index(v), :] = upd[:, :, k]
    res = TrackResult(n=n, T=T_, dyn_vars=dyn_t, tv_vars=tv, bins_tiled=None, values_tiled=tile(dense), init_bins=None,
                      init_values=Ti[:, 1:].T.contiguous(), attempts=None)
    xyz, good = S.integrate_tracks(model, res, opts=o, device=dev)
    torch.cuda.synchronize()
    t["integrate_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    text, off = S.format_tracks_csv(xyz, good)
    text, off = text.cpu().numpy(), off.cpu().numpy()
    t["format_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    Ti_h, z0, is_good = Ti.cpu().numpy(), xyz[2, 0].cpu().numpy(), good.cpu().numpy().astype(bool)
    view = memoryview(text)
    names_and_files(model, o, Ti_h, z0, is_good, T_, out_dir, lambda k: view[off[k]:off[k + 1]])
    t["write_s"] = time.perf_counter() - t0
    return t


def tree(root):
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            p = os.path.join(d, f)
            out[os.path.relpath(p, root)] = open(p, "rb").read()
    return out


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    path = materialize(tempfile.mkdtemp(prefix="emb_models_"), names=[MODEL])[MODEL]
    m = EncounterModel(path, idxZeroBoundaries=(1, 2, 3))
    lib = L.lib()
    out = {"gpu": gpu, "model": MODEL, "n": N, "T": T}

    # ---- the parser on the 1e5 x 600 transition.txt body
    res = m.sample_tracks(N, T, seed=42, device="cuda", want_bins=False)
    _, _, text, _ = m.format_em_sample(None, res.values_tiled, T, n=N)
    cols = 2 + len(m.temporal_map)
    vals = S.parse_table(text, cols)
    rows = int(vals.shape[0])
    o = _opts()
    got, bad = C.c_int64(), C.c_int64()

    def parse():
        L.check(lib.emb_parse_table(text.data_ptr(), len(text), cols, C.byref(o), rows, vals.data_ptr(), C.byref(got), C.byref(bad)))

    ref = vals.clone()
    t_parse = timed(parse)
    t_parse_helper = timed(lambda: S.parse_table(text, cols))
    assert torch.equal(vals, ref)
    split = kernel_split(parse, r"k_(?:parse|scan)_\w+")
    kernel_ms = sum(split.values())
    out["parse"] = {"text_bytes": len(text), "rows": rows, "cols": cols, "call_ms": t_parse, "parse_table_helper_ms": t_parse_helper,
                    "per_kernel_ms": split, "kernel_ms_total": kernel_ms,
                    "text_GB_per_s_of_call": len(text) / (t_parse["median"] / 1e3) / 1e9,
                    "text_GB_per_s_of_kernel_time": len(text) / (kernel_ms / 1e3) / 1e9 if kernel_ms else None}
    del vals, ref, text
    torch.cuda.empty_cache()

    # ---- the CSV formatter on the integrated 1e5 x 600 tracks
    xyz, good = S.integrate_tracks(m, res, device="cuda")
    del res
    ctext, coff = S.format_tracks_csv(xyz, good)
    total = C.c_int64()

    def fmt():
        L.check(lib.emb_format_tracks_csv(N, T, xyz.data_ptr(), good.data_ptr(), C.byref(o), len(ctext), ctext.data_ptr(),
                                          coff.data_ptr(), C.byref(total)))

    cref = ctext.clone()
    t_fmt = timed(fmt)
    t_fmt_helper = timed(lambda: S.format_tracks_csv(xyz, good))
    assert torch.equal(ctext, cref)
    split = kernel_split(fmt, r"k_(?:format_csv|scan)\w*")
    kernel_ms = sum(split.values())
    pin = torch.empty(len(ctext), dtype=torch.uint8, pin_memory=True)
    t_d2h = timed(lambda: pin.copy_(ctext, non_blocking=True))
    out["format_csv"] = {"text_bytes": len(ctext), "good_tracks": int(good.sum()), "call_ms": t_fmt,
                         "format_tracks_csv_helper_ms": t_fmt_helper, "per_kernel_ms": split, "kernel_ms_total": kernel_ms,
                         "text_GB_per_s_of_kernel_time": len(ctext) / (kernel_ms / 1e3) / 1e9 if kernel_ms else None,
                         "d2h_pinned_ms": t_d2h, "d2h_GB_per_s": len(ctext) / (t_d2h["median"] / 1e3) / 1e9}
    del xyz, good, ctext, coff, cref, pin
    torch.cuda.empty_cache()

    # ---- the file-to-file driver at n = 1e4, T = 600
    d = tempfile.mkdtemp(prefix="emb_s2t_")
    fi, ft = os.path.join(d, "initial.txt"), os.path.join(d, "transition.txt")
    em_sample(path, fi, ft, num_initial_samples=N_FILES, num_transition_samples=T, rng_seed=42)
    warm = os.path.join(d, "warm")
    S.sample2track(path, fi, ft, out_dir_parent=warm)   # warm-up: modules, allocator
    shutil.rmtree(warm)
    t0 = time.perf_counter()
    S.sample2track(path, fi, ft, out_dir_parent=os.path.join(d, "dev"))
    wall_dev = time.perf_counter() - t0
    dev_tree = tree(os.path.join(d, "dev"))
    shutil.rmtree(os.path.join(d, "dev"))
    split_dev = device_driver_split(path, fi, ft, os.path.join(d, "dev"))
    same_split = tree(os.path.join(d, "dev")) == dev_tree
    shutil.rmtree(os.path.join(d, "dev"))
    split_host = host_driver_split(path, fi, ft, os.path.join(d, "host"))
    host_tree = tree(os.path.join(d, "host"))
    shutil.rmtree(os.path.join(d, "host"))
    out["sample2track_n1e4"] = {
        "n": N_FILES, "T": T, "input_bytes": os.path.getsize(fi) + os.path.getsize(ft), "files": len(dev_tree),
        "output_bytes": sum(len(v) for v in dev_tree.values()),
        "trees_identical": dev_tree == host_tree and same_split,
        "wall_s_device_driver": wall_dev, "wall_s_device_driver_stages": split_dev, "stage_sum_s_device": sum(split_dev.values()),
        "wall_s_host_driver_stages": split_host, "stage_sum_s_host": sum(split_host.values())}
    shutil.rmtree(d)
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "sample2track_b200.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
