#!/usr/bin/env python
"""bench.py -- the measurement contract (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[2] per-GPU shard -- UncorEncounterModel.sample on
`uncor_allcode_fwsingle_v1.txt`, 1.25e6 tracks x 600 s per GPU (10M tracks over 8 GPUs; weak scaling).
A "step" is one pass of the hot path (emb_sample_tracks: initial network, 599 transition steps, 600
resample gates, de-discretisation, dense compact outputs) over one batch of 1.25e6 tracks.
  value : track-timesteps/s over all ranks, outputs resident in HBM (CUDA events, max over ranks)
  e2e   : same metric through the reference-facing call (UncorEncounterModel.sample's out_inits + sparse out_events, the
          reference's own track representation) via the C ABI with pinned HOST buffers, D2H inside the timed region;
          e2e_dense: the dense compact tiles of `value` copied to host memory instead
  roofline / cpu_baseline : see the task statement; cpu_baseline = oracle/oracle_c.c ("port") on host cores
The model tables (about 1 MB) are read-only inputs that legitimately live in L2; every step writes a
fresh 14.5 GB of outputs (>> 126 MB L2) with a new seed, so no step can reuse another's cache lines.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MODEL = "uncor_allcode_fwsingle_v1"
TRACKS_PER_GPU = 1_250_000
T = 600
# SURVEY.md 8(d): bytes(track) = T*n_dyn*(1+4) + n_initial*(1+4) + 4*(sum r_initial + sum r_dyn)
ALGO_BYTES_PER_TRACK = T * 3 * 5 + 7 * 5 + 4 * (39 + 19)
ALGO_BYTES_PER_UNIT = ALGO_BYTES_PER_TRACK / T          # 15.445 B per track-timestep at T = 600


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


DUMP_TRACKS = 2048        # tracks written whole by --dump-outputs: about 35 MB at T = 600


def tiled_tracks(buf, nvar, T, idx):
    """Tracks `idx` of a dense tiled output buffer as (k, nvar, T), read in place: TrackResult.bins / .values would untile
    all of it ([ceil(T/4)][ceil(n/128)][nvar][128][4], model.untile) into a 14 GB temporary first."""
    from em_model_manned_bayes_b200.model import TRACK_TILE
    nch = (T + 3) // 4
    a = buf.reshape(nch, -1, nvar, TRACK_TILE, 4)[:, idx // TRACK_TILE, :, idx % TRACK_TILE, :]      # (k, nch, nvar, 4)
    return a.permute(0, 2, 1, 3).reshape(len(idx), nvar, nch * 4)[:, :, :T]


def dump_outputs(out_dir, res, hist_initial, hist_transition):
    """--dump-outputs: what the last timed step returned to its caller, as <out_dir>/<name>.npy in float32 or float64.
    The full outputs are 14.5 GB, so a fixed seeded sample of DUMP_TRACKS tracks is written (every variable, every
    second; their indices in track_index.npy), together with the verification histograms, which cover every track."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(res.n, size=min(DUMP_TRACKS, res.n), replace=False))
    t = torch.from_numpy(idx).to(res.bins_tiled.device)
    arrays = {
        "track_index": idx.astype(np.float64),
        "bins": tiled_tracks(res.bins_tiled, len(res.dyn_vars), res.T, t).float(),   # (k, n_dyn, T), 1-based
        "values": tiled_tracks(res.values_tiled, len(res.tv_vars), res.T, t),         # (k, n_tv, T)
        "init_bins": res.init_bins[:, t].float(),                                      # (n_initial, k)
        "init_values": res.init_values[:, t],                                          # (n_initial, k)
        "attempts": (res.attempts[t].to(torch.int32) & 0xFFFF).float(),                 # uint16 held in an int16 tensor
        "hist_initial": hist_initial.double(),
        "hist_transition": hist_transition.double(),
    }
    arrays = {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def materialise_model():
    from em_model_manned_bayes_b200.model_archive import materialize
    d = os.path.join(tempfile.gettempdir(), "emb_bench_models_%d" % os.getuid())
    return materialize(d, names=[MODEL])[MODEL]


def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which is not what the CPU arm is about)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_port(path, n_tracks, threads):
    """Time oracle/oracle_c.c on `threads` host threads over n_tracks x T; returns track-timesteps/s."""
    import ctypes as C
    from oracle.c_oracle import COracle, lib
    from oracle.em_read import em_read
    co = COracle(em_read(path), uncor=True)
    import numpy as np
    ib = np.zeros((n_tracks, 7), dtype=np.int8)
    lib().oc_sample_tracks(C.byref(co.m), 1, 0, min(n_tracks, 256), T, threads, ib.ctypes.data, None, None, None, None, None)
    t0 = time.perf_counter()
    rc = lib().oc_sample_tracks(C.byref(co.m), 1, 0, n_tracks, T, threads, ib.ctypes.data, None, None, None, None, None)
    dt = time.perf_counter() - t0
    assert rc == 0
    return n_tracks * T / dt, dt


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation (the oracle's C port -- the
    reference itself is MATLAB and cannot run here) on all host threads, same config/metric/unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    path = materialise_model()
    per_thread = 30000
    n = per_thread * threads
    cpu_port(path, min(n, 512), threads)
    vals, t_all = [], 0.0
    for _ in range(args.warmup):
        cpu_port(path, max(256, n // 8), threads)
    for _ in range(args.steps):
        v, dt = cpu_port(path, n, threads)
        vals.append(v)
        t_all += dt
    value = n * T * args.steps / t_all
    sample = "%d tracks x %d s per step (%d per thread), oracle/oracle_c.c, OpenMP" % (n, T, per_thread)
    print(json.dumps({
        "impl": "reference", "metric": "sampled track-timesteps/sec", "value": value, "unit": "track-timesteps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "UncorEncounterModel.sample, %s, %d tracks x %d s per GPU (bounded CPU sample: %s)"
                   % (MODEL, TRACKS_PER_GPU, T, sample)},
        "cpu_baseline": {"value": value, "unit": "track-timesteps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "track-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--tracks", type=int, default=TRACKS_PER_GPU, help="tracks per GPU per step")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the B200 path only")
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from em_model_manned_bayes_b200 import _lib as L
    from em_model_manned_bayes_b200.model import UncorEncounterModel, async_status
    from em_model_manned_bayes_b200.shard import allreduce_histograms

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    if world > 1:
        # NCCL may print its version banner on stdout at init; the contract is ONE JSON line on stdout
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(dev))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    n = args.tracks
    lib = L.lib()
    path = materialise_model()
    m = UncorEncounterModel(path)
    hi = torch.zeros((m.n_initial, 64), dtype=torch.int64, device=dev)
    ht = torch.zeros((m.n_dyn, 64), dtype=torch.int64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm -------------------------------------------------------------------
    res = m.sample_compact(n, T, seed=1, first_sample=rank * n, device=dev)           # allocates outputs once
    for w in range(args.warmup):
        m.sample_compact(n, T, seed=100 + w, first_sample=rank * n, device=dev, out=res, enqueue_only=True)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = lib.emb_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for k in range(args.steps):
        last = k == args.steps - 1
        # enqueue_only: the passes run back to back on the stream (no host round trip per step); the status is collected below
        m.sample_compact(n, T, seed=1000 + k, first_sample=rank * n, device=dev, out=res, enqueue_only=True,
                         hist_initial=hi if last else None, hist_transition=ht if last else None)
        ev[k + 1].record()
    allreduce_histograms(hi, ht)          # the single collective of the job (verification only)
    barrier()
    async_status(local)                   # raises if any pass exhausted its rejection loop
    launches = lib.emb_launch_count() - launches0          # kernels of libemb200.so inside the timed region
    clk = clocks.stop() if rank == 0 else None
    total_ms = ev[0].elapsed_time(ev[-1])
    kern_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    units_per_step = world * n * T
    value = units_per_step * args.steps / (total_ms * 1e-3)
    assert int(hi.sum().item()) == world * n * m.n_initial, "verification histogram lost samples"
    assert int(ht.sum().item()) == world * n * (T - 1) * m.n_dyn
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, hi, ht)

    # ---- end-to-end arm: C ABI with pinned host buffers, D2H inside the timed region --------------
    nb = int(lib.emb_tracks_bins_len(m._h, n, T))
    nv = int(lib.emb_tracks_values_len(m._h, n, T))
    h_bins = torch.empty(nb, dtype=torch.int8).pin_memory()
    h_vals = torch.empty(nv, dtype=torch.float32).pin_memory()
    h_iv = torch.empty((m.n_initial, n), dtype=torch.float64).pin_memory()
    from em_model_manned_bayes_b200.model import TrackResult
    host_out = TrackResult(n=n, T=T, dyn_vars=res.dyn_vars, tv_vars=res.tv_vars, bins_tiled=h_bins, values_tiled=h_vals,
                           init_bins=None, init_values=h_iv, attempts=None)
    del res
    torch.cuda.empty_cache()
    o = m.uncor_opts()
    o.mem, o.device = L.EMB_MEM_HOST, local
    m.sample_tracks(n, T, seed=5, first_sample=rank * n, opts=o, out=host_out)      # warm-up (allocations, page faults)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.e2e_steps):
        m.sample_tracks(n, T, seed=2000 + k, first_sample=rank * n, opts=o, out=host_out)
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = units_per_step * args.e2e_steps / float(t.item())
    d2h = nb + nv * 4 + h_iv.numel() * 8 + 4
    del h_bins, h_vals, host_out

    # ---- end-to-end, sparse contract: the reference's own track representation (out_events) ------------
    # emb_sample_track_events with pinned host buffers: count pass, prefix sum, write pass, D2H of rows + offsets + inits
    probe = m.sample_events(n, T, seed=6, first_sample=rank * n, opts=m.uncor_opts(), device=dev, want_init=False)
    cap = int(probe.total * 1.03)
    del probe
    torch.cuda.empty_cache()
    h_words = torch.empty(cap, dtype=torch.int32).pin_memory()      # packed rows: 4 + 1 bytes (emb_sample_track_events_packed)
    h_dts = torch.empty(cap, dtype=torch.uint8).pin_memory()
    h_off = torch.empty(n + 1, dtype=torch.int64).pin_memory()
    import ctypes as C
    tot = C.c_int64(0)
    init_only = L.TrackOut(None, None, None, h_iv.data_ptr(), None, None, None)

    def events_call(seed):
        rng = L.Rng(seed, rank * n)
        L.check(lib.emb_sample_track_events_packed(m._h, C.byref(rng), n, T, C.byref(o), cap, h_words.data_ptr(), h_dts.data_ptr(),
                                                   h_off.data_ptr(), C.byref(init_only), C.byref(tot)))
    for k in range(max(6, args.warmup)):      # warm-up calls: the first one also fills the library's device memory pool
        events_call(7 + k)
    barrier()
    ev_steps = []
    t0 = time.perf_counter()
    ev_n = 2 * args.e2e_steps          # 40 ms steps: twice as many as the 300 ms dense steps
    for k in range(ev_n):
        t1 = time.perf_counter()
        events_call(3000 + k)
        ev_steps.append((time.perf_counter() - t1) * 1e3)
    barrier()
    ev_s = time.perf_counter() - t0
    t = torch.tensor([ev_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_events_value = units_per_step * ev_n / float(t.item())
    ev_d2h = int(tot.value) * 5 + (n + 1) * 8 + h_iv.numel() * 8 + 12

    # ---- the other single-GPU configuration of BASELINE.json, for the record (rank 0, device-resident) -----
    other = {}
    if rank == 0:
        from em_model_manned_bayes_b200.model import EncounterModel
        from em_model_manned_bayes_b200.model_archive import materialize
        # configs[0]: the reference's own CPU-sized case, 1,000 tracks x 300 s on uncor_1200code_v2p1, through the reference-facing
        # call with host buffers (launch- and latency-bound: three small kernels, two syncs and the D2H of ~100 rows per track)
        p0 = materialize(os.path.join(tempfile.gettempdir(), "emb_bench_models_%d" % os.getuid()),
                         names=["uncor_1200code_v2p1"])["uncor_1200code_v2p1"]
        m0 = UncorEncounterModel(p0)
        o0 = m0.uncor_opts()
        o0.mem, o0.device = L.EMB_MEM_HOST, local
        n0, T0 = 1000, 300
        ev0 = torch.empty(400 * n0, dtype=torch.int64).pin_memory()
        off0 = torch.empty(n0 + 1, dtype=torch.int64).pin_memory()
        iv0 = torch.empty((m0.n_initial, n0), dtype=torch.float64).pin_memory()
        init0 = L.TrackOut(None, None, None, iv0.data_ptr(), None, None, None)
        tot0 = C.c_int64(0)

        def call0(seed):
            rng = L.Rng(seed, 0)
            L.check(lib.emb_sample_track_events(m0._h, C.byref(rng), n0, T0, C.byref(o0), ev0.numel(), ev0.data_ptr(),
                                                off0.data_ptr(), C.byref(init0), C.byref(tot0)))
        for k in range(5):
            call0(k)
        t0 = time.perf_counter()
        for k in range(50):
            call0(10 + k)
        dt0 = (time.perf_counter() - t0) / 50
        other["configs[0] uncor_1200code_v2p1, 1,000 tracks x 300 s, UncorEncounterModel.sample outputs in host memory"] = {
            "value": n0 * T0 / dt0, "unit": "track-timesteps/s", "ms_per_call": dt0 * 1e3}
        del m0
        gp = materialize(os.path.join(tempfile.gettempdir(), "emb_bench_models_%d" % os.getuid()), names=["glider_v1"])["glider_v1"]
        g = EncounterModel(gp)
        n2 = 100_000_000
        buf = g.sample_initial(n2, seed=1, device=dev, want_values=False, want_attempts=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for k in range(3):
            g.sample_initial(n2, seed=2 + k, device=dev, want_values=False, want_attempts=False, out=buf, enqueue_only=True)
        e1.record()
        torch.cuda.synchronize()
        async_status(local)
        del buf
        other["configs[1] glider_v1 initial network only, 100M samples, int8 bins"] = {
            "value": 3 * n2 / (e0.elapsed_time(e1) * 1e-3), "unit": "samples/s"}
        # the same with the de-discretised values (bn_sample + dediscretize): SURVEY 8d counts 5*(1+4) = 25 B per sample -- the
        # compact contract (emb_sample_initial_f32: int8 bin + fp32 value per variable), and the fp64 values of out_inits
        for key, kw, written in (("int8 bins + fp32 values", dict(values_fp32=True), 25.0), ("int8 bins + fp64 values", {}, 45.0)):
            buf = g.sample_initial(n2, seed=1, device=dev, want_values=True, want_attempts=False, **kw)
            torch.cuda.synchronize()
            e0.record()
            for k in range(3):
                g.sample_initial(n2, seed=2 + k, device=dev, want_values=True, want_attempts=False, out=buf, enqueue_only=True, **kw)
            e1.record()
            torch.cuda.synchronize()
            async_status(local)
            del buf
            v2 = 3 * n2 / (e0.elapsed_time(e1) * 1e-3)
            other["configs[1] glider_v1 initial network only, 100M samples, " + key] = {
                "value": v2, "unit": "samples/s", "algorithmic_bytes_per_unit": 25.0, "written_bytes_per_unit": written,
                "roofline_frac": v2 * 25.0 / 1e9 / peaks()[0]}
        del g
        torch.cuda.empty_cache()

        def timed(fn, reps=3):
            fn(0)
            torch.cuda.synchronize()
            e0.record()
            for k in range(reps):
                fn(1 + k)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e-3 / reps

        # configs[3]: correlated model (cor_v2p1.txt is missing from the public checkout -> cor_v1.txt, 16 initial + 4 dynamic
        # variables, dbn_sample.m slow branch), 10M encounters x 60 s (em_sample.m:26)
        mdir = os.path.join(tempfile.gettempdir(), "emb_bench_models_%d" % os.getuid())
        cp = materialize(mdir, names=["cor_v1"])["cor_v1"]
        cm = EncounterModel(cp)
        n4, T4 = 10_000_000, 60
        r4 = cm.sample_tracks(n4, T4, seed=1, device=dev)
        dt = timed(lambda k: cm.sample_tracks(n4, T4, seed=10 + k, device=dev, out=r4, enqueue_only=True))
        async_status(local)
        other["configs[3] cor_v1 (stand-in for the missing cor_v2p1), 10M encounters x 60 s, dense compact outputs"] = {
            "value": n4 * T4 / dt, "unit": "track-timesteps/s", "ms": dt * 1e3,
            # SURVEY 8d: 4*(1+4) B per step + (16*(1+4) + 4*(99+36)) B per track
            "algorithmic_bytes_per_unit": 20.0 + (80.0 + 540.0) / T4,
            "roofline_frac": n4 * T4 / dt * (20.0 + 620.0 / T4) / 1e9 / peaks()[0]}
        del r4, cm
        torch.cuda.empty_cache()

    # ---- configs[4]: CorTerminalModel, 1M encounters PER GPU (weak scaling like the main workload), every rank -------------
    # geometry sampling (sample.m) + four trajectory chains per encounter (createEncounter.m) on synthetic trajectory DBNs of
    # the documented layout (the 20 model files are missing upstream); sharded by encounter index: rank r owns encounters
    # [r*n5, (r+1)*n5), both kernels keyed by the global index (first_sample), no collective on the data path
    from em_model_manned_bayes_b200.model import CorTerminalModel
    from em_model_manned_bayes_b200.model_archive import materialize as _mat
    from em_model_manned_bayes_b200.synthetic import write_terminal_model_set
    mdir5 = os.path.join(tempfile.gettempdir(), "emb_bench_models_%d" % os.getuid())
    tp_ = _mat(mdir5, names=["terminal_v3_radar_encounter_model"])["terminal_v3_radar_encounter_model"]
    write_terminal_model_set(os.path.join(mdir5, "traj"))
    tm = CorTerminalModel(tp_, parameters_directory=os.path.join(mdir5, "traj"))
    n5, tmax5 = 1_000_000, 120
    vals5, _, _ = tm.sample_raw(n5, seed=1, first_sample=rank * n5, device=dev)
    geo = vals5.T.contiguous()
    r5 = tm.create_encounters(geo, tmax5, seed=2, first_sample=rank * n5, device=dev)
    e5 = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    reps5 = 3
    barrier()
    e5[0].record()
    for k in range(reps5):
        tm.sample_raw(n5, seed=20 + k, first_sample=rank * n5, device=dev)
    e5[1].record()
    for k in range(reps5):
        tm.create_encounters(geo, tmax5, seed=30 + k, first_sample=rank * n5, device=dev, out=r5)
    e5[2].record()
    barrier()
    t5 = torch.tensor([e5[0].elapsed_time(e5[1]) / reps5, e5[1].elapsed_time(e5[2]) / reps5], dtype=torch.float64, device=dev)
    st5 = r5.len.to(torch.int64).sum().reshape(1)
    if world > 1:
        dist.all_reduce(t5, op=dist.ReduceOp.MAX)           # device time: max over ranks
        dist.all_reduce(st5, op=dist.ReduceOp.SUM)          # trajectory states of the whole job
    dt_geo, dt_traj, states = float(t5[0]) * 1e-3, float(t5[1]) * 1e-3, int(st5.item())
    config4 = {"value": states / dt_traj, "unit": "trajectory states/s", "ms_chains": dt_traj * 1e3, "ms_geometry": dt_geo * 1e3,
               "encounters_per_s": world * n5 / (dt_traj + dt_geo), "encounters": world * n5, "n_gpus": world, "scaling": "weak",
               "states_per_encounter": states / (world * n5),
               # 5 fp32 fields per state written; the chains are bound by the latency of their per-lane column gathers and fp64 chains, not by HBM (DESIGN.md section 5)
               "algorithmic_bytes_per_unit": 20.0, "roofline_frac": states / dt_traj * 20.0 / 1e9 / (peaks()[0] * world)}
    del r5, geo, vals5, tm
    torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    other["configs[4] CorTerminalModel 1M encounters per GPU: sample (geometry) + createEncounter chains, tmax 120 s, synthetic "
          "trajectory DBNs, sharded by encounter index"] = config4
    peak, peak_src = peaks()
    k_ms = statistics.mean(kern_ms)
    achieved = ALGO_BYTES_PER_UNIT * n * T / (k_ms * 1e-3) / 1e9
    traffic = None      # dram__bytes_read.sum + dram__bytes_write.sum per unit from the committed ncu --set full capture
    issue = None        # the limiter the ncu capture names: warp-instructions issued against the schedulers' peak
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get("bytes_per_unit") * n * T
            # smsp__inst_executed.sum / (units / 32) of the same capture; one warp-instruction per scheduler per clock is the
            # issue peak: SMs x 4 schedulers x the SM clock sampled during the timed region
            sms = torch.cuda.get_device_properties(local).multi_processor_count
            mhz = (clk or {}).get("sm_mhz") or (clk or {}).get("sm_max_mhz") or 1965.0
            wi = float(tj["warp_inst_per_warp_unit"])
            issue = {"warp_inst_per_32_units": wi, "issue_peak_per_s": sms * 4 * mhz * 1e6,
                     "frac": (n * T / 32.0) * wi / (k_ms * 1e-3) / (sms * 4 * mhz * 1e6),
                     "pipes_pct": tj.get("pipes_pct"), "source": tj.get("source")}
        except Exception:
            traffic = None
    out = {
        "metric": "sampled track-timesteps/sec", "value": value, "unit": "track-timesteps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "UncorEncounterModel.sample (BASELINE configs[2] per-GPU shard): %s, %d tracks x %d s per GPU, "
                               "start all-free, prior 0, dense compact outputs (int8 bins of 3 dynamic variables + fp32 "
                               "values of 4 time-varying variables)" % (MODEL, n, T),
                   "cache": "each step writes %.1f GB of fresh outputs (>> L2); the 1 MB model tables are the only re-read input"
                            % ((nb + nv * 4) / 1e9),
                   "sharding": "global sample index, rank r owns [r*n, (r+1)*n); one NCCL all-reduce of verification histograms"},
        # e2e = the reference-facing call: UncorEncounterModel.sample's outputs (out_inits + the sparse out_events lists the
        # reference itself returns, UncorEncounterModel.m:253-300) through emb_sample_track_events with pinned HOST buffers
        "e2e": {"value": e2e_events_value, "unit": "track-timesteps/s", "h2d_bytes_per_step": 3400,
                "d2h_bytes_per_step": ev_d2h, "steps": ev_n,
                "ms_per_step": [round(x, 2) for x in ev_steps],
                "d2h_bytes_per_unit": ev_d2h / (n * T),
                "contract": "UncorEncounterModel.sample outputs: sparse out_events rows (5-byte packed rows: dt, variable, bin and the "
                            "23 value bits; the host evaluates dediscretize.m:39 in fp64) + offsets + out_inits in host memory, "
                            "emb_sample_track_events_packed (count pass, prefix sum, write pass, D2H inside the timed region)"},
        "e2e_dense": {"value": e2e_value, "unit": "track-timesteps/s", "h2d_bytes_per_step": 3400, "d2h_bytes_per_step": d2h,
                      "steps": args.e2e_steps,
                      "contract": "dense compact tiles in host memory (the same emb_sample_tracks call as `value`); PCIe-bound at 19.0 B/unit"},
        "other_configs": other,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_unit": ALGO_BYTES_PER_UNIT,
                     "written_bytes_per_unit": (nb + nv * 4) / (n * T), "kernel_ms": k_ms,
                     # the kernel is bound by instruction issue, not by HBM (DESIGN.md section 5): issue slots used / peak
                     "issue_frac": issue["frac"] if issue else None, "issue": issue},
        "clocks": clk,
    }
    n1_file = os.path.join(tempfile.gettempdir(), "emb_bench_e2e_n1_%d.json" % os.getuid())
    if world == 1:
        try:
            json.dump({"e2e": e2e_events_value, "value": value, "tracks": n}, open(n1_file, "w"))
        except OSError:
            pass
        out["e2e"]["efficiency_vs_n1"] = 1.0
    else:   # weak-scaling efficiency of the end-to-end number against the N=1 run of the same box (driver runs 1,2,4,8 in turn)
        try:
            n1 = json.load(open(n1_file))
            out["e2e"]["efficiency_vs_n1"] = e2e_events_value / (world * n1["e2e"]) if n1.get("tracks") == n else None
            out["efficiency_vs_n1"] = value / (world * n1["value"]) if n1.get("tracks") == n else None
        except (OSError, ValueError, KeyError):
            out["e2e"]["efficiency_vs_n1"] = None
    if world == 1 and not args.no_cpu:
        threads = host_threads()
        ntr = 80000 * threads
        v, dt = cpu_port(path, ntr, threads)
        out["cpu_baseline"] = {"value": v, "unit": "track-timesteps/s", "cores": threads, "kind": "port",
                               "sample": "%d tracks x %d s, oracle/oracle_c.c (plain-C restatement of the MATLAB path), OpenMP, %.1f s"
                                         % (ntr, T, dt)}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
