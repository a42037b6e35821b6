"""Times of the em_sample text formatter (emb_format_em_sample): initial.txt and transition.txt formatted on the device.

    python tools/time_format.py [OUT_DIR]        (default profiles/)

Workloads (cor_v1, bench.py configs[3] per-GPU shard: 1.25M tracks x 60 s):
  - emb_sample_tracks of the shard into device memory (CUDA events, median of 10 calls after a warm-up);
  - emb_format_em_sample of its output, both texts, inputs and outputs device-resident, capacities from a sizing call: the
    whole call (CUDA events, median of 10), EncounterModel.format_em_sample as em_sample calls it (allocation of upper-bound
    buffers included), and its kernels split into count pass, prefix sum and write pass (torch.profiler
    with CUDA activities over 10 more calls, in a separate window; per-call medians of the kernel times);
  - the D2H copy of both texts into pinned host memory (CUDA events, median of 10);
  - em_sample writing both files to local disk at n = 1e5, T = 60, wall clock: the device formatter against the host loop that
    em_sample.py ran before it (kept below as the comparison), on the same sample_tracks output.  The files must be identical.
Writes format_b200.json into OUT_DIR with the card name and power limit read in the same run (nvidia-smi's read-only query).
"""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from em_model_manned_bayes_b200 import _lib as L  # noqa: E402
from em_model_manned_bayes_b200.em_sample import em_sample  # noqa: E402
from em_model_manned_bayes_b200.model import EncounterModel  # noqa: E402
from em_model_manned_bayes_b200.model_archive import materialize  # noqa: E402

MODEL, N, T = "cor_v1", 1_250_000, 60


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
    return times[len(times) // 2], times[0]


def em_sample_host_loop(path, fi_name, ft_name, n, T, rng_seed=42, chunk=1 << 16):
    """em_sample.py's formatting before the device formatter: sample on the device, copy the dense values to the host, format
    every number with Python's '%g'.  Kept here only as the comparison."""
    parms = EncounterModel(path, idxZeroBoundaries=(1, 2, 3))
    tv = list(parms.timevarying_vars)
    cols = [tv.index(int(v)) for v in parms.temporal_map[:, 0]]
    with open(fi_name, "w", encoding="utf-8") as fi, open(ft_name, "w", encoding="utf-8") as ft:
        fi.write("id " + "".join("%s " % l for l in parms.labels_initial) + "\n")
        ft.write("initial_id t " + "".join("%s " % parms.labels_transition[int(k) - 1] for k in parms.temporal_map[:, 1]) + "\n")
        for first in range(0, n, chunk):
            m = min(chunk, n - first)
            res = parms.sample_tracks(m, T, seed=rng_seed, first_sample=first, device="cuda", want_bins=False)
            iv = res.init_values.cpu().numpy().T
            vals = res.values.cpu().numpy().astype(np.float64)[:, cols, :]
            for k in range(m):
                ii = first + k + 1
                fi.write("%d " % ii + " ".join("%g" % x for x in iv[k]) + "\n")
                rows = vals[k].T
                ft.write("".join("%g %g " % (ii, j) + " ".join("%g" % x for x in rows[j]) + "\n" for j in range(T)))


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    path = materialize(tempfile.mkdtemp(prefix="emb_models_"), names=[MODEL])[MODEL]
    m = EncounterModel(path, idxZeroBoundaries=(1, 2, 3))
    lib = L.lib()
    res = m.sample_tracks(N, T, seed=42, device="cuda", want_bins=False)
    t_sample = timed(lambda: m.sample_tracks(N, T, seed=42, device="cuda", want_bins=False, out=res))

    ti, oi, tt, ot = m.format_em_sample(res, first_id=1)
    o = m._opts()
    o.mem, o.device, o.stream = L.EMB_MEM_DEVICE, torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream
    iv, vt = res.init_values, res.values_tiled
    totals = (C.c_int64 * 2)()

    def call():
        L.check(lib.emb_format_em_sample(m._h, N, T, 1, iv.data_ptr(), vt.data_ptr(), C.byref(o), len(ti), ti.data_ptr(),
                                         oi.data_ptr(), len(tt), tt.data_ptr(), ot.data_ptr(), totals))

    ref_i, ref_t = ti.clone(), tt.clone()
    t_format = timed(call)
    t_python = timed(lambda: m.format_em_sample(res, first_id=1))   # what em_sample runs: one call into upper-bound buffers
    assert torch.equal(ti, ref_i) and torch.equal(tt, ref_t)
    text_bytes = len(ti) + len(tt)

    from torch.profiler import ProfilerActivity, profile
    reps = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and ("k_format" in e.name or "k_scan" in e.name):
            name = re.search(r"k_(?:format|scan)_\w+", e.name).group(0)
            kern.setdefault(name, []).append(e.device_time if hasattr(e, "device_time") else e.cuda_time)
    per = {k: float(np.median(v)) / 1000.0 for k, v in kern.items()}   # us -> ms, per launch
    scans = sum(v for k, v in per.items() if "k_scan" in k) * 2        # one prefix sum of each text
    split = {"count_pass_ms": per.get("k_format_initial_count", 0.0) + per.get("k_format_transition_count", 0.0),
             "prefix_sum_ms": scans,
             "write_pass_ms": per.get("k_format_initial", 0.0) + per.get("k_format_transition", 0.0),
             "per_kernel_ms": per}
    kernel_ms = split["count_pass_ms"] + split["prefix_sum_ms"] + split["write_pass_ms"]

    pin = torch.empty(text_bytes, dtype=torch.uint8, pin_memory=True)

    def d2h():
        pin[:len(ti)].copy_(ti, non_blocking=True)
        pin[len(ti):].copy_(tt, non_blocking=True)

    t_d2h = timed(d2h)

    del res, ti, tt, oi, ot, ref_i, ref_t
    torch.cuda.empty_cache()
    n_small = 100_000
    d = tempfile.mkdtemp(prefix="emb_format_files_")
    f = [os.path.join(d, x) for x in ("i_new.txt", "t_new.txt", "i_old.txt", "t_old.txt")]
    em_sample(path, f[0], f[1], num_initial_samples=20, num_transition_samples=T)   # warm-up
    t0 = time.perf_counter()
    em_sample(path, f[0], f[1], num_initial_samples=n_small, num_transition_samples=T, rng_seed=42)
    wall_new = time.perf_counter() - t0
    t0 = time.perf_counter()
    em_sample_host_loop(path, f[2], f[3], n_small, T)
    wall_old = time.perf_counter() - t0
    same = all(open(a, "rb").read() == open(b, "rb").read() for a, b in ((f[0], f[2]), (f[1], f[3])))
    file_bytes = os.path.getsize(f[0]) + os.path.getsize(f[1])
    for x in f:
        os.remove(x)

    out = {
        "gpu": gpu,
        "model": MODEL, "n": N, "T": T,
        "text_bytes": text_bytes, "initial_bytes": int(totals[0]), "transition_bytes": int(totals[1]),
        "sample_tracks_ms": {"median": t_sample[0], "min": t_sample[1]},
        "format_call_ms": {"median": t_format[0], "min": t_format[1]},
        "format_em_sample_python_ms": {"median": t_python[0], "min": t_python[1]},
        "format_kernels": split,
        "format_kernel_ms_total": kernel_ms,
        "text_bytes_per_s_of_kernel_time": text_bytes / (kernel_ms / 1e3) if kernel_ms else None,
        "d2h_pinned_ms": {"median": t_d2h[0], "min": t_d2h[1]},
        "d2h_bytes_per_s": text_bytes / (t_d2h[0] / 1e3),
        "formatting_cheaper_than_d2h": kernel_ms < t_d2h[0],
        "em_sample_n1e5": {"n": n_small, "T": T, "file_bytes": file_bytes, "files_identical": same,
                           "wall_s_device_formatter": wall_new, "wall_s_host_loop": wall_old},
    }
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "format_b200.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
