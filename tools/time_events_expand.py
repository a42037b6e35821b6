"""Times of the event-list expansion (emb_track_events_expand[_packed]): out_samples and the out_EME control rows on the device.

    python tools/time_events_expand.py [OUT_DIR]        (default profiles/)

Workloads (uncor_allcode_fwsingle_v1, the out_EME spec):
  - controls only, 1.25M x 600 s, packed and 8-byte rows, inputs and outputs device-resident: one call = count pass, prefix
    sum, the total to the host, write pass (CUDA events, median of 10 calls after a warm-up).  Bytes per track are what the
    call must move: the rows twice (the count pass reads the dt of every row), offsets twice, init_values, the counts and
    offsets it writes and reads, and the control rows; compared with a device-to-device copy of 4 GB timed in the same run.
  - samples plus controls, 1e5 x 600 s, device-resident (3.4 GB of fp64 samples).
  - the host-buffer chain, 1e5 x 600 s: sample_events_packed into host memory, then expand_events_gpu on host buffers (the
    library stages them), wall clock; against model.py's expand_events + controls_of on the 8-byte rows of the same lists on
    this host's CPU.
Every device result is checked against the others (packed against 8-byte controls times, samples of the chain against the
CPU expansion) before it is timed.  Writes events_expand_b200.json into OUT_DIR with the card name and power limit read in the
same run (nvidia-smi's read-only query).
"""
import ctypes as C
import json
import math
import os
import platform
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from em_model_manned_bayes_b200 import _lib as L  # noqa: E402
from em_model_manned_bayes_b200.model import UncorEncounterModel, controls_of, expand_events  # noqa: E402
from em_model_manned_bayes_b200.model_archive import materialize  # noqa: E402

MODEL = "uncor_allcode_fwsingle_v1"


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


def device_call(m, res, packed, spec, samples, rows, ctl_off):
    """one emb_track_events_expand[_packed] call on device buffers (capacity = rows.shape[0])"""
    o = m._opts()
    o.mem, o.device, o.stream = L.EMB_MEM_DEVICE, torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream
    total = C.c_int64(0)
    ptr = lambda t: None if t is None else t.data_ptr()
    lib = L.lib()

    def call():
        if packed:
            rc = lib.emb_track_events_expand_packed(m._h, res.n, res.T, ptr(res.init_values), ptr(res.words), ptr(res.dts),
                                                    ptr(res.offsets), C.byref(o), C.byref(spec), ptr(samples), rows.shape[0],
                                                    ptr(rows), ptr(ctl_off), C.byref(total))
        else:
            rc = lib.emb_track_events_expand(m._h, res.n, res.T, ptr(res.init_values), ptr(res.events), ptr(res.offsets),
                                             C.byref(o), C.byref(spec), ptr(samples), rows.shape[0], ptr(rows), ptr(ctl_off),
                                             C.byref(total))
        L.check(rc)
    return call


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles")
    os.makedirs(out_dir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(gpu, flush=True)
    m = UncorEncounterModel(materialize(tempfile.mkdtemp(), names=[MODEL])[MODEL])
    ni = m.n_initial
    vars_, mul, div = m.out_eme_spec()
    spec = L.ControlsSpec()
    spec.n_cols = 3
    for j in range(3):
        spec.vars[j], spec.mul[j], spec.div[j] = vars_[j], mul[j], div[j]
    src = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms_copy, _ = timed(lambda: dst.copy_(src))
    copy_bw = 2 * src.numel() / (ms_copy * 1e-3)
    del src, dst
    res = {"gpu": gpu, "copy_bandwidth_TBps": copy_bw / 1e12, "host_cpu": "%s, %d logical CPUs" % (platform.processor() or
           platform.machine(), os.cpu_count()), "workloads": {}}

    # ---- controls only, 1.25M x 600 s, device-resident ------------------------------------------------------------------
    n, T = 1_250_000, 600
    o = m.uncor_opts()
    pk = m.sample_events_packed(n, T, seed=1, opts=o, device="cuda")
    ev = m.sample_events(n, T, seed=1, opts=m.uncor_opts(), device="cuda")
    w = {"n": n, "T": T, "rows_per_track": pk.total / n}
    outs = {}
    for name, r, packed, row_bytes, dt_bytes in (("packed", pk, True, 5, 5), ("rows8", ev, False, 8, 4)):
        _, c = m.expand_events_gpu(r, spec=(vars_, mul, div), want_samples=False)
        outs[name] = c
        total = int(c.rows.shape[0])
        rows = torch.empty_like(c.rows)
        ctl_off = torch.empty_like(c.offsets)
        fn = device_call(m, r, packed, spec, None, rows, ctl_off)
        fn()
        assert torch.equal(rows, c.rows) and torch.equal(ctl_off, c.offsets)
        nbytes = (r.total * (row_bytes + dt_bytes) + 2 * 8 * (n + 1) + 8 * ni * n + 4 * n * 2 + 2 * 8 * (n + 1)
                  + 8 * 4 * total)
        ms, best = timed(fn)
        w[name] = {"ms_median": ms, "ms_best": best, "control_rows_per_track": total / n, "bytes": nbytes,
                   "bytes_per_track": nbytes / n, "TBps": nbytes / (ms * 1e-3) / 1e12,
                   "fraction_of_copy_bw": nbytes / (ms * 1e-3) / copy_bw}
        print(name, json.dumps(w[name]), flush=True)
    assert torch.equal(outs["packed"].offsets, outs["rows8"].offsets)
    assert torch.equal(outs["packed"].rows[:, 0], outs["rows8"].rows[:, 0])
    res["workloads"]["controls only, %s 1.25M x 600 s, device-resident" % MODEL] = w
    del pk, ev, outs, rows, ctl_off
    torch.cuda.empty_cache()

    # ---- samples plus controls, 1e5 x 600 s, device-resident -------------------------------------------------------------
    n = 100_000
    pk = m.sample_events_packed(n, T, seed=2, opts=m.uncor_opts(), device="cuda")
    smp, c = m.expand_events_gpu(pk, spec=(vars_, mul, div))
    rows, ctl_off = torch.empty_like(c.rows), torch.empty_like(c.offsets)
    samples = torch.empty_like(smp)
    fn = device_call(m, pk, True, spec, samples, rows, ctl_off)
    fn()
    assert torch.equal(samples, smp) and torch.equal(rows, c.rows)
    nbytes = samples.numel() * 8 + rows.numel() * 8 + pk.total * 10 + 8 * ni * n + 40 * (n + 1)
    ms, best = timed(fn)
    res["workloads"]["samples + controls, %s 1e5 x 600 s, device-resident, packed rows" % MODEL] = w = {
        "n": n, "T": T, "ms_median": ms, "ms_best": best, "samples_GB": samples.numel() * 8 / 1e9, "bytes": nbytes,
        "TBps": nbytes / (ms * 1e-3) / 1e12, "fraction_of_copy_bw": nbytes / (ms * 1e-3) / copy_bw}
    print("samples + controls", json.dumps(w), flush=True)
    del pk, smp, c, rows, ctl_off, samples
    torch.cuda.empty_cache()

    # ---- the host-buffer chain against the CPU expansion, 1e5 x 600 s ------------------------------------------------------
    chain = []
    for _ in range(3):
        t0 = time.perf_counter()
        pk = m.sample_events_packed(n, T, seed=3, opts=m.uncor_opts())
        t1 = time.perf_counter()
        hs, hc = m.expand_events_gpu(pk, spec=(vars_, mul, div))
        t2 = time.perf_counter()
        chain.append((t2 - t0, t1 - t0, t2 - t1))
    chain.sort()
    ev = m.sample_events(n, T, seed=3, opts=m.uncor_opts())
    assert np.array_equal(np.asarray(ev.offsets), np.asarray(pk.offsets))
    e = np.asarray(ev.events)
    t0 = time.perf_counter()
    dense = expand_events(np.ascontiguousarray(ev.init_values.T), e["dt"], e["var"], e["value"], ev.offsets, T)
    ctl = controls_of(dense, e["dt"], ev.offsets, [v - 1 for v in vars_])
    for c in ctl:
        c[:, 1] /= 60.0
        c[:, 2] *= math.pi / 180.0
        c[:, 3] *= 1.68780972222222
    t_cpu = time.perf_counter() - t0
    assert np.array_equal(np.concatenate(ctl)[:, 0], hc.rows[:, 0])
    res["workloads"]["host-buffer chain, %s 1e5 x 600 s" % MODEL] = w = {
        "n": n, "T": T, "gpu_chain_s_median": chain[1][0], "gpu_sample_packed_s": chain[1][1], "gpu_expand_s": chain[1][2],
        "cpu_expand_events_controls_of_s": t_cpu, "speedup": t_cpu / chain[1][0],
        "note": "GPU chain: sample_events_packed to host memory, then expand_events_gpu on host buffers (samples + out_EME "
                "controls, staged through the library); CPU: expand_events + controls_of + the out_EME scaling on the 8-byte "
                "rows of the same lists"}
    print("host chain", json.dumps(w), flush=True)
    with open(os.path.join(out_dir, "events_expand_b200.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
