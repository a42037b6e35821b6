"""Kernel times of the event-list scoring (emb_loglik_track_events[_packed]) against the dense scoring (emb_loglik_tracks) of the
same tracks, all inputs device-resident and larger than L2 (CUDA events after a warm-up, median of 10 calls).

    python tools/time_loglik_events.py [OUT_DIR]        (default profiles/)

Workloads: the flagship tracks (uncor_allcode_fwsingle_v1, 1.25M x 600 s, frozen parents), cor_v1 10M x 60 s (per-step parents)
and the flagship tracks with correct_dbn (per-step).  Each is sampled three times with one seed -- 8-byte rows, packed rows,
dense tiles: the same tracks -- and each form is scored in the same run; the results are checked equal (frozen: bit for bit,
per-step: 1e-12 relative) before they are timed.  Bytes per track are what each call must read (8 or 5 bytes per row plus the
offsets, or the tiles; init bins) and write (two fp64), compared with the copy bandwidth measured in the same run (a
device-to-device copy of 4 GB).  Writes loglik_events_b200.json and, from a separate torch.profiler pass,
loglik_events_profile.txt into OUT_DIR; prints the card name and power limit (nvidia-smi's read-only query) with the numbers.
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
    print(gpu, flush=True)
    import tempfile
    models = materialize(tempfile.mkdtemp())
    src = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms_copy, _ = timed(lambda: dst.copy_(src))
    copy_bw = 2 * src.numel() / (ms_copy * 1e-3)
    del src, dst
    res = {"gpu": gpu, "copy_bandwidth_TBps": copy_bw / 1e12, "workloads": {}}
    calls = {}

    def workload(name, model, n, T, seed, correct_dbn):
        m = EncounterModel(models[model])
        ni = m.n_initial
        w = {"n": n, "T": T, "correct_dbn": correct_dbn, "frozen": not m.is_dynvar_depend and not correct_dbn}
        tr = m.sample_tracks(n, T, seed=seed, device="cuda", want_values=False)
        forms = {"dense": (lambda: m.loglik_tracks(tr, correct_dbn=correct_dbn), tr.bins_tiled.numel() + ni * n + 16 * n)}
        ev = m.sample_events(n, T, seed=seed, device="cuda")
        w["rows_per_track"] = ev.total / n
        forms["rows8"] = (lambda: m.loglik_events(ev, correct_dbn=correct_dbn), 8 * ev.total + 8 * (n + 1) + ni * n + 16 * n)
        if len(m.gated_vars) <= 7 and T <= 1023:
            pk = m.sample_events_packed(n, T, seed=seed, device="cuda")
            forms["packed"] = (lambda: m.loglik_events(pk, correct_dbn=correct_dbn), 5 * pk.total + 8 * (n + 1) + ni * n + 16 * n)
        di, dt = forms["dense"][0]()
        for f in ("rows8", "packed"):
            if f not in forms:
                continue
            gi, gt = forms[f][0]()
            assert torch.equal(gi, di), (name, f, "initial term")
            if w["frozen"]:
                assert torch.equal(gt, dt), (name, f, "transition term")
            else:
                fin = torch.isfinite(dt)
                assert torch.equal(fin, torch.isfinite(gt)) and torch.equal(gt[~fin], dt[~fin]), (name, f, "-inf terms")
                rel = ((gt[fin] - dt[fin]).abs() / dt[fin].abs().clamp_min(1e-300)).max().item()
                assert rel <= 1e-12, (name, f, rel)
                w[f + "_max_rel_vs_dense"] = rel
        for f, (fn, nbytes) in forms.items():
            ms, best = timed(fn)
            w[f] = {"ms_median": ms, "ms_best": best, "bytes": nbytes, "bytes_per_track": nbytes / n,
                    "TBps": nbytes / (ms * 1e-3) / 1e12, "fraction_of_copy_bw": nbytes / (ms * 1e-3) / copy_bw}
            calls[name + " " + f] = fn
        w["speedup_rows8_vs_dense"] = w["dense"]["ms_median"] / w["rows8"]["ms_median"]
        if "packed" in w:
            w["speedup_packed_vs_dense"] = w["dense"]["ms_median"] / w["packed"]["ms_median"]
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        return tr, ev

    keep = workload("uncor_allcode_fwsingle_v1 1.25M x 600 s", "uncor_allcode_fwsingle_v1", 1_250_000, 600, 1, False)
    keep += workload("cor_v1 10M x 60 s", "cor_v1", 10_000_000, 60, 2, False)
    keep += workload("uncor_allcode_fwsingle_v1 1.25M x 600 s correct_dbn", "uncor_allcode_fwsingle_v1", 1_250_000, 600, 1, True)
    with open(os.path.join(out_dir, "loglik_events_b200.json"), "w") as f:
        json.dump(res, f, indent=1)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for fn in calls.values():
            fn()
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=20)
    with open(os.path.join(out_dir, "loglik_events_profile.txt"), "w") as f:
        f.write(gpu + "\n" + table + "\n")
    print(table)


if __name__ == "__main__":
    main()
