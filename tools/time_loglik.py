"""Kernel times of the log-likelihood entry points on device-resident inputs larger than L2 (CUDA events after a warm-up).

    python tools/time_loglik.py [OUT_DIR]        (default profiles/)

Workloads: the flagship fast-branch tracks (uncor_allcode_fwsingle_v1, 1.25M x 600 s, 2.25 GB of tiles), per-step tracks (cor_v1,
10M x 60 s) and glider initial states (1e8 samples).  For each: ms per call, bytes the call must move (tile and init-bin reads,
fp64 writes), and that over the copy bandwidth measured in the same run (a device-to-device copy of 4 GB).  Writes
loglik_b200.json and, from a separate torch.profiler pass, loglik.pt.trace.json into OUT_DIR; prints the card name and power limit
(nvidia-smi's read-only query) with the numbers.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from em_model_manned_bayes_b200.model import EncounterModel  # noqa: E402
from em_model_manned_bayes_b200.model_archive import materialize  # noqa: E402


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


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles")
    os.makedirs(out_dir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    import tempfile
    models = materialize(tempfile.mkdtemp())
    # copy bandwidth of this card: read + write of a 4 GB buffer
    src = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms_copy, _ = timed(lambda: dst.copy_(src))
    copy_bw = 2 * src.numel() / (ms_copy * 1e-3)
    del src, dst
    res = {"gpu": gpu, "copy_bandwidth_TBps": copy_bw / 1e12, "workloads": {}}

    def record(name, ms, best, bytes_moved, units, unit_name):
        res["workloads"][name] = {"ms_median": ms, "ms_best": best, "bytes": bytes_moved, "bytes_per_" + unit_name: bytes_moved / units,
                                  unit_name + "s_per_s": units / (ms * 1e-3), "TBps": bytes_moved / (ms * 1e-3) / 1e12,
                                  "fraction_of_copy_bw": bytes_moved / (ms * 1e-3) / copy_bw}
        print(name, json.dumps(res["workloads"][name]), flush=True)

    calls = {}
    # fast branch: 1.25M x 600 s
    m = EncounterModel(models["uncor_allcode_fwsingle_v1"])
    n, T = 1_250_000, 600
    tr = m.sample_tracks(n, T, seed=1, device="cuda", want_values=False)
    calls["fast"] = lambda: m.loglik_tracks(tr)
    ms, best = timed(calls["fast"])
    record("uncor_allcode_fwsingle_v1 tracks 1.25M x 600 s (frozen parents)", ms, best,
           tr.bins_tiled.numel() + tr.init_bins.numel() + 16 * n, n * T, "track_second")
    # per-step branch: cor_v1 10M x 60 s
    mc = EncounterModel(models["cor_v1"])
    nc, Tc = 10_000_000, 60
    tc = mc.sample_tracks(nc, Tc, seed=2, device="cuda", want_values=False)
    calls["step"] = lambda: mc.loglik_tracks(tc)
    ms, best = timed(calls["step"])
    record("cor_v1 tracks 10M x 60 s (per-step parents)", ms, best, tc.bins_tiled.numel() + tc.init_bins.numel() + 16 * nc,
           nc * Tc, "track_second")
    # glider initial states, 1e8
    mg = EncounterModel(models["glider_v1"])
    ng = 100_000_000
    gb, _, _ = mg.sample_initial(ng, seed=3, device="cuda", want_values=False, want_attempts=False)
    calls["initial"] = lambda: mg.loglik_initial(gb)
    ms, best = timed(calls["initial"])
    record("glider_v1 initial states 1e8", ms, best, gb.numel() + 8 * ng, ng, "sample")

    with open(os.path.join(out_dir, "loglik_b200.json"), "w") as f:
        json.dump(res, f, indent=1)
    # kernel names and times from a separate profiled pass (one call each)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for fn in calls.values():
            fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(out_dir, "loglik.pt.trace.json"))
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=15)
    with open(os.path.join(out_dir, "loglik_profile.txt"), "w") as f:
        f.write(gpu + "\n" + table + "\n")
    print(table)


if __name__ == "__main__":
    main()
