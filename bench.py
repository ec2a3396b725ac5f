#!/usr/bin/env python
"""Benchmark of the per-planning-step assessment hot path (BASELINE.json metric:
trajectory x agent x step evaluations / s; p50 per-planning-step latency).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c-sweep|c-lat]
                    [--dump-outputs DIR]

One "step" = one pass of the dense metric core over the whole synthetic sweep bundle
(C-sweep: 1,000,000 trajectories x 256 phantom agents x 50 steps, all seven metrics), split by
trajectory over the ranks in interleaved blocks (strong scaling, total work fixed) followed by ONE
in-place all-gather of the per-trajectory result vectors when N > 1.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from frenetix_occlusion_b200 import synthetic as S  # noqa: E402

METRIC = "traj_agent_step_evals_per_s"
UNIT = "evals/s"
CHUNK = 125_000          # trajectories per generation chunk (8 chunks = the 1 M sweep)

# ALGORITHMIC work per evaluation (DESIGN.md "Roofline"; SURVEY.md 8(d)):
#   F(g, c) = 300 + 1050*g flop per (trajectory, agent, step) evaluation, g = fraction of evaluations
#   inside the 5 m CP gate; plus BE: per colliding pair ~6 bisection probes x T steps x 60 flop.
F_BASE, F_CP, F_BE_STEP = 300.0, 1050.0, 60.0
# EXECUTED work model (what the kernel really evaluates after its exact bounds; counts from fo_metric_stats):
# bounds per visited evaluation (squared centre distance, squared speed difference, 5 m gate), exact oriented-box
# distance, LR4S impact-angle logit, collision probability (36 Phi), BE probe step.
FX_BOUNDS, FX_OBB, FX_LR4S, FX_CP, FX_BE_STEP = 30.0, 170.0, 90.0, 1050.0, 60.0
FX_WINDOW = 16.0         # one (agent, 8-step window) box test of the window filter
FP32_LANES_PER_SM = 128            # FP32 FMA lanes per SM: peak = SMs x 128 x 2 flop x max SM clock (theoretical, fixed)
SHARD_BLOCK = 1024                 # trajectories per interleaved shard block (N > 1)


def bench_config(wl):
    """The workload description both arms print (identical dicts: the driver compares them)."""
    return {"workload": wl["name"], "n_traj": wl["n_traj"], "n_agents": wl["n_agents"], "n_steps": wl["n_states"] - 1,
            "metrics": "all7"}


def workload(name):
    if name == "c-lat":
        return dict(S.C_LAT)
    return dict(S.C_SWEEP)


def gen_ego(n_traj, n_states, first_chunk, keep=None):
    """Deterministic global bundle: chunk k of CHUNK trajectories is seeded with SEED + 100 + k.  ``keep`` (sorted global
    indices) selects the rows of an interleaved shard while the chunks are generated one after the other."""
    if keep is not None:
        out = np.empty((len(keep), n_states, 5), dtype=np.float32)
        done = 0
        for k in range((n_traj + CHUNK - 1) // CHUNK):
            lo, hi = k * CHUNK, min(n_traj, (k + 1) * CHUNK)
            sel = keep[(keep >= lo) & (keep < hi)] - lo
            if len(sel):
                out[done:done + len(sel)] = S.ego_bundle(hi - lo, n_states, seed=S.SEED + 100 + k)[sel].astype(np.float32)
                done += len(sel)
        return out
    out = np.empty((n_traj, n_states, 5), dtype=np.float32)
    done, k = 0, first_chunk
    while done < n_traj:
        m = min(CHUNK, n_traj - done)
        out[done:done + m] = S.ego_bundle(m, n_states, seed=S.SEED + 100 + k).astype(np.float32)
        done += m
        k += 1
    return out


def make_case(wl, n_traj, first_chunk=0, keep=None):
    return {"dt": 0.1, "vehicle": {k: float(S._f32(v)) for k, v in S.VEHICLE.items()},
            "ego": gen_ego(n_traj, wl["n_states"], first_chunk, keep=keep),
            "agents": S.agent_table(wl["n_agents"], wl["n_states"], seed=S.SEED + 1),
            "activated_metrics": list(S.ALL_METRICS), "thresholds": dict(S.DEFAULT_THRESHOLDS)}


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        while self.ok and not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def _oracle_chunk(args):
    case, lo, hi = args
    from oracle import metric_oracle as MO
    sub = dict(case)
    sub["ego"] = np.asarray(case["ego"][lo:hi], dtype=np.float64)
    out = MO.evaluate_bundle(sub, want_detail=False)
    return int(out["valid"].sum())


def cpu_oracle_throughput(wl, n_traj_sample, cores, steps=1, warmup=0):
    """Times the CPU restatement of the path (oracle B, float64 numpy -- the reference itself needs
    shapely/commonroad/frenetix and cannot be installed here) on ``cores`` processes."""
    import multiprocessing as mp
    case = make_case(wl, n_traj_sample)
    bounds = np.linspace(0, n_traj_sample, cores + 1).astype(int)
    jobs = [(case, int(bounds[i]), int(bounds[i + 1])) for i in range(cores) if bounds[i + 1] > bounds[i]]
    evals = n_traj_sample * wl["n_agents"] * (wl["n_states"] - 1)
    times = []
    ctx = mp.get_context("fork")
    with ctx.Pool(len(jobs)) as pool:
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(_oracle_chunk, jobs)
            t1 = time.perf_counter()
            if it >= warmup:
                times.append(t1 - t0)
    sec = float(np.mean(times))
    return evals / sec, sec, evals


def run_reference(args):
    """--impl reference: the path's CPU implementation on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workload(args.workload)
    cores = os.cpu_count() or 1
    n_sample = min(wl["n_traj"], 64 * cores if wl["n_agents"] >= 128 else 1000)
    value, sec, evals = cpu_oracle_throughput(wl, n_sample, cores, steps=args.steps, warmup=args.warmup)
    sample = (f"{n_sample} of {wl['n_traj']} trajectories x {wl['n_agents']} agents x {wl['n_states'] - 1} steps per step, "
              f"oracle B (vectorised float64 numpy port of the reference metrics) on {cores} processes")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(wl),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "sample_traj": n_sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine, BundleResult
    from frenetix_occlusion_b200.parallel import PeerResultGatherer, ResultGatherer, shard_indices

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    wl = workload(args.workload)
    N_total, A, T = wl["n_traj"], wl["n_agents"], wl["n_states"]
    # trajectory shard of this rank (strong scaling): interleaved blocks, so every rank gets the same mix of cheap and
    # expensive trajectories whatever the order of the bundle
    if world > 1:
        mine = shard_indices(N_total, world, rank, SHARD_BLOCK)
        n_local = len(mine)
        case = make_case(wl, N_total, keep=mine)
    else:
        n_local = N_total
        case = make_case(wl, n_local)
    ego_host = torch.from_numpy(case["ego"]).pin_memory()

    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"], device=dev)
    eng.set_agents(AgentSet.from_case(case["agents"]))
    ego_dev = ego_host.to(dev)
    # N > 1: the kernel writes valid / summary / flags straight into this rank's slice of the gather buffer -- of EVERY
    # rank's buffer when they are peer-mapped (fused exchange: the epilogue's stores cross NVLink, no all-gather
    # follows); --exchange nccl keeps the in-place all_gather_into_tensor
    gatherer, exchange = None, "none"
    if world > 1:
        if args.exchange == "peer":
            ok = torch.ones(1, dtype=torch.int32, device=dev)
            try:
                gatherer = PeerResultGatherer(N_total, L.FO_SUMMARY_K, dev, block=SHARD_BLOCK)
                exchange = "peer"
            except Exception as e:  # noqa: BLE001  (IPC not permitted on this box: every rank falls back together)
                sys.stderr.write(f"rank {rank}: peer-mapped exchange unavailable ({e}); using the NCCL all-gather\n")
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                gatherer = None
        if gatherer is None:
            gatherer = ResultGatherer(N_total, L.FO_SUMMARY_K, dev, block=SHARD_BLOCK)
            exchange = "nccl"
    if gatherer is not None:
        out = gatherer.local_result()
        assert out.valid.shape[0] == n_local
    else:
        out = BundleResult(torch.empty(n_local, dtype=torch.uint8, device=dev),
                           torch.empty((n_local, L.FO_SUMMARY_K), dtype=torch.float32, device=dev),
                           torch.empty(n_local, dtype=torch.int32, device=dev))
    host_valid = torch.empty(n_local, dtype=torch.uint8).pin_memory()
    host_summary = torch.empty((n_local, L.FO_SUMMARY_K), dtype=torch.float32).pin_memory()
    host_flags = torch.empty(n_local, dtype=torch.int32).pin_memory()

    def step_out():
        return gatherer.local_result() if gatherer is not None else out   # peer exchange: two buffers alternate

    def step_resident():
        eng.assess(ego_dev, out=step_out())
        if world > 1:   # the single exchange step of the path: all-gather, or the handshake of the fused form
            gatherer.gather()

    # e2e on the torch path (N > 1): the shard crosses PCIe in geometrically growing chunks on a copy stream while
    # the previous chunk is evaluated (same schedule as fo_metric_bundle_host), then the single all-gather and D2H
    traj_bytes = T * 5 * 4
    bounds, at, stepn = [0], 0, max(1, (16 << 20) // traj_bytes)
    while at < n_local:
        at = min(n_local, at + stepn)
        bounds.append(at)
        stepn *= 4
    copy_stream = torch.cuda.Stream(device=dev)
    chunk_events = [torch.cuda.Event() for _ in bounds[1:]]
    stage_dev = torch.empty_like(ego_dev)
    chunk_cache = {}

    def chunks_of(o):
        if id(o) not in chunk_cache:
            mk = gatherer.slice_of if gatherer is not None else (lambda r, lo, hi: BundleResult(r.valid[lo:hi], r.summary[lo:hi], r.flags[lo:hi]))
            chunk_cache[id(o)] = (o, [mk(o, lo, hi) for lo, hi in zip(bounds[:-1], bounds[1:])])
        return chunk_cache[id(o)][1]

    def step_e2e():
        out = step_out()
        chunk_out = chunks_of(out)
        cur = torch.cuda.current_stream(dev)
        copy_stream.wait_stream(cur)                      # the staging buffer is free again
        with torch.cuda.stream(copy_stream):
            for c, (lo, hi) in enumerate(zip(bounds[:-1], bounds[1:])):
                stage_dev[lo:hi].copy_(ego_host[lo:hi], non_blocking=True)   # H2D from pinned memory
                chunk_events[c].record(copy_stream)
        for c, (lo, hi) in enumerate(zip(bounds[:-1], bounds[1:])):
            cur.wait_event(chunk_events[c])
            eng.assess(stage_dev[lo:hi], out=chunk_out[c])
        if world > 1:
            gatherer.gather()
        host_valid.copy_(out.valid, non_blocking=True)   # D2H of the step's result
        host_summary.copy_(out.summary, non_blocking=True)
        host_flags.copy_(out.flags, non_blocking=True)
        cur.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sample_clocks=False, per_step_events=False):
        for _ in range(warmup):
            fn()
        barrier()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler is not None and sampler.ok:
            sampler.start()
        launches0 = L.lib.fo_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kern = []
        e0.record()
        for _ in range(steps):
            if per_step_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                eng.assess(ego_dev, out=step_out())
                b.record()
                kern.append((a, b))
                if world > 1:
                    gatherer.gather()
            else:
                fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = L.lib.fo_launch_count() - launches0
        clocks = sampler.stop() if sampler is not None else None
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        kern_ms = [a.elapsed_time(b) for a, b in kern]
        return ms, launches, clocks, kern_ms

    evals_total = N_total * A * (T - 1)
    ms, launches, clocks, kern_ms = timed(step_resident, args.steps, args.warmup, sample_clocks=True, per_step_events=True)
    value = evals_total * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # what the last timed step returned, taken before the e2e calls below write into the same buffers, so that two
        # builds can be compared output for output.  flags (u32 bit masks) go to float64, which holds every value
        # exactly; C-sweep writes 4 + 40 + 8 MB.  The files hold finite numbers only, and the summary's special values
        # map without loss: +inf (min_dce / wttc when there is none) becomes the float32 maximum, which no real value
        # reaches, and NaN (the two BE columns of a trajectory flagged FO_F_BE_RANGE, as flags.npy records) becomes 0
        if gatherer is not None:
            gatherer.current_result()
            valid, summary, flags = gatherer.assembled()          # global trajectory order
        else:
            valid, summary, flags = out.valid, out.summary, out.flags
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t, dtype in (("valid", valid, np.float32), ("summary", summary, np.float32), ("flags", flags, np.float64)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.nan_to_num(t.cpu().numpy().astype(dtype)))
    e2e_how = ""
    if world == 1:
        # the reference-facing C-ABI call with HOST buffers: fo_metric_bundle_host copies the bundle and the raw
        # predictions to the device, packs the agent table, runs the kernel, copies valid/summary/flags back and
        # synchronises -- timed with the host clock around the blocking call
        import ctypes as C
        ag = eng.agents
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)  # noqa: E731
        keep = [f32(ag.x), f32(ag.y), f32(ag.yaw), f32(ag.v), f32(ag.var_x), f32(ag.var_y),
                np.ascontiguousarray(ag.n_states, dtype=np.int32), np.ascontiguousarray(ag.kind, dtype=np.int32),
                f32(ag.length), f32(ag.width), f32(ag.buf_length), f32(ag.buf_width)]
        raw = L.FoAgentsRaw()
        raw.n_agents, raw.t_stride = ag.n_agents, ag.t_stride
        (raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y, raw.n_states, raw.kind, raw.length, raw.width,
         raw.buf_length, raw.buf_width) = [a.ctypes.data for a in keep]
        prm = eng._args(ego_dev, out)

        def step_capi():
            L.check(L.lib.fo_metric_bundle_host(C.c_void_p(ego_host.data_ptr()), n_local, T, C.byref(raw), C.byref(prm),
                                                C.c_void_p(host_valid.data_ptr()), C.c_void_p(host_summary.data_ptr()),
                                                C.c_void_p(host_flags.data_ptr()), None, None), "fo_metric_bundle_host")

        for _ in range(max(1, args.warmup // 2)):
            step_capi()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_capi()
        ms_e2e = (time.perf_counter() - t0) * 1e3
        assert bool((host_valid.to(dev) == out.valid).all()), "C-ABI host call and device-resident call disagree"
        e2e_how = "fo_metric_bundle_host (C ABI, pinned host buffers in and out), host wall clock around the blocking call"
    else:
        # N > 1: the same C-ABI host call per rank; its device destinations are this rank's slice of the gather buffer (and,
        # fused, of every peer's), then the exchange step (handshake / all-gather).  Host wall clock, maximum over ranks.
        import ctypes as C
        ag = eng.agents
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)  # noqa: E731
        keep = [f32(ag.x), f32(ag.y), f32(ag.yaw), f32(ag.v), f32(ag.var_x), f32(ag.var_y),
                np.ascontiguousarray(ag.n_states, dtype=np.int32), np.ascontiguousarray(ag.kind, dtype=np.int32),
                f32(ag.length), f32(ag.width), f32(ag.buf_length), f32(ag.buf_width)]
        raw = L.FoAgentsRaw()
        raw.n_agents, raw.t_stride = ag.n_agents, ag.t_stride
        (raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y, raw.n_states, raw.kind, raw.length, raw.width,
         raw.buf_length, raw.buf_width) = [a.ctypes.data for a in keep]
        prm_cache = {}

        def step_capi_n():
            o = step_out()
            if id(o) not in prm_cache:
                prm_cache[id(o)] = (o, eng._args(ego_dev, o))
            prm = prm_cache[id(o)][1]
            L.check(L.lib.fo_metric_bundle_host(C.c_void_p(ego_host.data_ptr()), n_local, T, C.byref(raw), C.byref(prm),
                                                C.c_void_p(host_valid.data_ptr()), C.c_void_p(host_summary.data_ptr()),
                                                C.c_void_p(host_flags.data_ptr()), None, None), "fo_metric_bundle_host")
            gatherer.gather()
            torch.cuda.current_stream(dev).synchronize()

        for _ in range(max(1, args.warmup // 2)):
            step_capi_n()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_capi_n()
        ms_e2e = (time.perf_counter() - t0) * 1e3
        barrier()
        t = torch.tensor([ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
        assert bool((host_valid.to(dev) == gatherer.current_result().valid).all()), "host copy and gather buffer disagree"
        e2e_how = ("fo_metric_bundle_host per rank (C ABI, pinned host shard in, results into the gather buffer and back to "
                   "the host) + the exchange step, host wall clock, max over ranks")
        if args.e2e_torch:
            ms_e2e, _, _, _ = timed(step_e2e, args.steps, max(1, args.warmup // 2))
            e2e_how = "torch: pinned H2D (chunked, overlapped) + fo_metric_bundle + exchange + D2H, CUDA events, max over ranks"
    e2e_value = evals_total * args.steps / (ms_e2e * 1e-3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- workload statistics for the algorithmic flop count (sample of the same bundle, on the GPU) ----
    samp = min(n_local, 20000)
    st = eng.work_stats(ego_dev[:samp])
    ev = max(samp * A * (T - 1), 1)
    g_frac = st["cp"] / ev                                  # fraction of evaluations inside the 5 m CP gate
    be_pairs = st["be"] / max(samp * A, 1)                  # fraction of pairs with 0 < ttc < inf (BE work)
    flop_per_eval = F_BASE + F_CP * g_frac + be_pairs * 6 * T * F_BE_STEP / (T - 1)
    executed_flop_per_eval = (FX_BOUNDS * st["visited"] + FX_OBB * st["obb"] + FX_LR4S * st["lr4s"] + FX_CP * st["cp"]
                              + FX_BE_STEP * st["be_probes"] * T + FX_WINDOW * st.get("windows", 0)) / ev

    # ---- peaks: FP32 = the fixed theoretical FMA peak of this GPU (SMs x 128 lanes x 2 flop x max SM clock; no measured
    # FP32 figure exists in MEASURED_PEAKS.json), with the library's own FFMA probe beside it for information; HBM = the
    # driver-measured copy bandwidth
    import ctypes as C
    props = torch.cuda.get_device_properties(dev)
    sm_max_mhz = float((clocks or {}).get("sm_max_mhz") or 1965.0)
    peak_tflops = props.multi_processor_count * FP32_LANES_PER_SM * 2 * sm_max_mhz * 1e6 / 1e12
    peak_src = (f"theoretical, fixed: {props.multi_processor_count} SMs x {FP32_LANES_PER_SM} FP32 lanes x 2 flop x "
                f"{sm_max_mhz:.0f} MHz (max SM clock from NVML)")
    ms_p, fl_p = C.c_float(), C.c_double()
    probe_tflops = None
    if L.lib.fo_probe_fp32_peak(200000, C.byref(ms_p), C.byref(fl_p), None) == 0 and ms_p.value > 0:
        probe_tflops = fl_p.value / (ms_p.value * 1e-3) / 1e12
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "of measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "of fallback 6.65 TB/s"

    # DRAM traffic of the dominant kernel: ncu --set full capture of the same launch shape, committed under profiles/
    # (a profiler cannot run inside the timed region); the file and the commit that last touched it are named
    traffic, traffic_src = None, None
    try:
        import subprocess
        tf = os.path.join("profiles", "traffic_r2.json")
        if not os.path.exists(os.path.join(ROOT, tf)):
            tf = os.path.join("profiles", "traffic_r1.json")
        with open(os.path.join(ROOT, tf)) as f:
            tr = json.load(f)
        if wl["name"] == "C-sweep":
            traffic = int(tr["traffic"] * (n_local / 1_000_000))
            h = subprocess.run(["git", "-C", ROOT, "log", "-1", "--format=%h", "--", tf], capture_output=True, text=True).stdout.strip()
            traffic_src = f"{tf} (commit {h or 'n/a'}): {tr['source']}; dram__bytes_read.sum + dram__bytes_write.sum per launch"
    except Exception:
        pass

    k_ms = float(np.mean(kern_ms)) if kern_ms else ms / args.steps
    evals_local = n_local * A * (T - 1)
    effective_tflops = evals_local * flop_per_eval / (k_ms * 1e-3) / 1e12
    executed_tflops = evals_local * executed_flop_per_eval / (k_ms * 1e-3) / 1e12
    alg_bytes = n_local * (T * 5 * 4 + 1 + 4 + 4 * L.FO_SUMMARY_K) + A * T * 32
    roofline = {"bound": "fp32", "kernel": "fo_metric_sweep_kernel",
                # what the FP32 pipe really does: flops of the work left after the kernel's exact bounds
                "achieved": executed_tflops, "peak": peak_tflops, "unit": "TFLOP/s", "frac": executed_tflops / peak_tflops,
                "peak_source": peak_src, "probe_tflops": probe_tflops, "kernel_ms": k_ms,
                "flop_per_eval_executed": executed_flop_per_eval,
                # the contract's algorithmic figure (SURVEY.md 8d: every evaluation charged at full cost)
                "effective_achieved": effective_tflops, "effective_frac": effective_tflops / peak_tflops,
                "flop_per_eval_algorithmic": flop_per_eval, "gate_fraction": g_frac, "be_pair_fraction": be_pairs,
                "traffic": traffic, "traffic_source": traffic_src,
                "executed": {"note": "work the kernel evaluates after its exact bounds (fo_metric_stats on a "
                                     f"{samp}-trajectory sample): fractions per (traj, agent, step) evaluation",
                             "obb_fraction": st["obb"] / ev, "lr4s_fraction": st["lr4s"] / ev, "cp_fraction": st["cp"] / ev,
                             "be_pairs_fraction": st["be"] / max(samp * A, 1),
                             "be_probes_per_pair": st["be_probes"] / max(st["be"], 1),
                             "visited_fraction": st["visited"] / ev,
                             "window_items_kept": st.get("windows_kept", 0) / max(st.get("windows", 0), 1)},
                "hbm": {"bound": "hbm", "achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": alg_bytes,
                        "peak_source": hbm_src},
                "note": "the summary kernel is instruction-issue bound (ncu: issue slots 84 % busy, FMA pipe 36 %, ALU 45 %, XU 22 %; profiles/ncu_r2_sweep_summary.txt), not "
                        "FP32- or HBM-bound: frac counts only flops it executes; effective_frac charges every "
                        "(traj, agent, step) evaluation at the algorithmic cost although exact bounds skip 80 % of them, "
                        "so it measures pruning, not pipe utilisation"}

    # ---- CPU baselines (rank 0, N = 1 only): the float64 port timed here on the box's cores, and the reference's own
    # metric code (oracle A), which can only run where the reference tree is (build container): committed measurement
    cpu, cpu_ref_code = None, None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        n_sample = min(N_total, 64 * cores if A >= 128 else 1000)
        reps = 8
        v, sec, _ = cpu_oracle_throughput(wl, n_sample, cores, steps=reps, warmup=1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n_sample} trajectories x {A} agents x {T - 1} steps, {reps} timed passes after one warm-up, "
                         f"oracle B (float64 numpy port of the reference metrics) on {cores} processes, "
                         f"{sec:.1f} s per pass"}
    try:
        with open(os.path.join(ROOT, "profiles", "oracle_a_cpu_r2.json")) as f:
            oa = json.load(f)
        w = oa["workloads"][wl["name"]]
        cpu_ref_code = {"value": w["all_cores"]["evals_per_s"], "unit": UNIT, "cores": w["all_cores"]["processes"],
                        "kind": "reference", "one_core_value": w["one_core"]["evals_per_s"],
                        "sample": f"{w['all_cores']['pairs']} (trajectory, agent) pairs x {T - 1} steps of {wl['name']}: {oa['what']}",
                        "where": oa["host"]["where"] + "; profiles/oracle_a_cpu_r2.json (scripts/time_oracle_a.py)"}
    except Exception:
        pass

    # ---- p50 latency of the per-planning-step case (C-lat, device resident, one launch) -----------------
    lat = None
    if not args.no_latency:
        lc = make_case(workload("c-lat"), 1000)
        eng_l = MetricEngine(lc["vehicle"], lc["dt"], lc["activated_metrics"], lc["thresholds"], device=dev)
        eng_l.set_agents(AgentSet.from_case(lc["agents"]))
        ego_l = torch.from_numpy(lc["ego"]).to(dev)
        out_l = eng_l.assess(ego_l)
        for _ in range(50):
            eng_l.assess(ego_l, out=out_l)
        torch.cuda.synchronize()
        ts = []
        for _ in range(1000):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng_l.assess(ego_l, out=out_l)
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        # the same launch replayed from a CUDA graph: no per-call host work between the events
        graph, _ = eng_l.capture(ego_l, out=out_l)
        for _ in range(50):
            graph.replay()
        torch.cuda.synchronize()
        tg = []
        for _ in range(1000):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            graph.replay()
            b.record()
            b.synchronize()
            tg.append(a.elapsed_time(b) * 1e3)
        # wall clock of the eager call including the host side (what a planner thread sees)
        tw = []
        for _ in range(300):
            t0 = time.perf_counter()
            eng_l.assess(ego_l, out=out_l)
            torch.cuda.synchronize()
            tw.append((time.perf_counter() - t0) * 1e6)
        # host side of one planning step: packing 1000 trajectory objects, and the pinned H2D copy of the bundle
        import types as _types
        from frenetix_occlusion_b200.adapter import BundlePacker
        objs = [_types.SimpleNamespace(cartesian=_types.SimpleNamespace(x=lc["ego"][q, :, 0], y=lc["ego"][q, :, 1],
                                                                        theta=lc["ego"][q, :, 2], v=lc["ego"][q, :, 3],
                                                                        a=lc["ego"][q, :, 4])) for q in range(1000)]
        packer = BundlePacker(1000, lc["ego"].shape[1])
        packer.pack(objs)
        t0 = time.perf_counter()
        for _ in range(5):
            staged = packer.pack(objs)
        pack_ms = (time.perf_counter() - t0) / 5 * 1e3
        # the planner's own SoA export (stacked [N, T] columns): no per-object Python work
        cols = [np.ascontiguousarray(lc["ego"][:, :, q]) for q in range(5)]
        packer.pack_columns(*cols)
        t0 = time.perf_counter()
        for _ in range(50):
            staged = packer.pack_columns(*cols)
        pack_cols_ms = (time.perf_counter() - t0) / 50 * 1e3
        # object -> result end to end for C-lat: pack columns + pinned H2D + one launch + D2H of valid
        host_v = torch.empty(1000, dtype=torch.uint8).pin_memory()
        te = []
        for _ in range(200):
            t0 = time.perf_counter()
            staged = packer.pack_columns(*cols)
            ego_l.copy_(staged, non_blocking=True)
            eng_l.assess(ego_l, out=out_l)
            host_v.copy_(out_l.valid, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            te.append((time.perf_counter() - t0) * 1e6)
        th = []
        for _ in range(200):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ego_l.copy_(staged, non_blocking=True)
            b.record()
            b.synchronize()
            th.append(a.elapsed_time(b) * 1e3)
        lat = {"workload": "C-lat 1000x32x30 all7 device-resident", "p50_us": float(np.percentile(ts, 50)),
               "adapter_pack_1000_objects_ms": pack_ms, "adapter_pack_columns_ms": pack_cols_ms,
               "columns_to_mask_e2e_p50_us": float(np.percentile(te, 50)),
               "h2d_620kB_pinned_p50_us": float(np.percentile(th, 50)),
               "p95_us": float(np.percentile(ts, 95)), "iters": 1000,
               "graph_p50_us": float(np.percentile(tg, 50)), "graph_p95_us": float(np.percentile(tg, 95)),
               "wall_p50_us": float(np.percentile(tw, 50)),
               "note": "p50_us: CUDA events around the eager ctypes call (includes host launch overhead while the GPU "
                       "idles); graph_p50_us: the same launch replayed from a CUDA graph; wall_p50_us: host wall "
                       "clock of call + synchronize"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": bench_config(wl),
            "run": {"parallelism": (f"interleaved trajectory shards ({SHARD_BLOCK}-trajectory blocks) x{world} + " +
                                    ("result exchange fused into the metric kernel: its epilogue stores [valid u8 | flags i32 | "
                                     "summary f32] into every rank's peer-mapped gather buffer over NVLink, then a 4-byte "
                                     "all-reduce as completion handshake" if exchange == "peer" else
                                     "1 in-place all_gather of [valid u8 | flags i32 | summary f32]")) if world > 1 else "single GPU",
                    "exchange": exchange,
                    "l2": "inputs (1.02 GB bundle) larger than L2, no flush needed" if N_total * T * 20 > 2.5e8
                          else "inputs smaller than L2 (latency case, resident by design)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n_local * T * 5 * 4) * world,
                    "d2h_bytes_per_step": int(n_local * (1 + 4 + 4 * L.FO_SUMMARY_K)) * world, "ms_per_step": ms_e2e / args.steps,
                    "how": e2e_how},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "cpu_baseline_reference_code": cpu_ref_code, "latency": lat}
    if not args.no_stages:
        try:
            line["stages"] = run_stages(dev, hbm_peak=hbm_peak, hbm_src=hbm_src, fp32_peak=peak_tflops, fp32_src=peak_src)
        except Exception as e:      # secondary numbers must never cost the headline line
            line["stages"] = {"error": repr(e)}
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_stages(dev, hbm_peak=6650.0, hbm_src="of fallback 6.65 TB/s", fp32_peak=74.4, fp32_src="theoretical"):
    """Secondary numbers of the other two stages of the path and of one whole planning cycle (rank 0 only)."""
    import random
    import torch
    from frenetix_occlusion_b200.visibility import raycast_frames
    from frenetix_occlusion_b200.prediction import rollout_cv
    out = {}
    # ---- stage 1, C-vis: 4096 rays x 512 rectangles per frame over 10 k frames (BASELINE.json configs[4]) ----
    F, R, O = S.C_VIS["n_frames"], S.C_VIS["n_rays"], S.C_VIS["n_obstacles"]
    rect = torch.from_numpy(S.obstacle_frames(F, O)).to(dev)
    flags = torch.ones((F, O), dtype=torch.uint8, device=dev)
    ego = torch.zeros((F, 3), dtype=torch.float32, device=dev)
    res = raycast_frames(ego, rect, flags, None, 50.0, 360.0, R, device=dev)
    for _ in range(3):
        raycast_frames(ego, rect, flags, None, 50.0, 360.0, R, device=dev, out=res)
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        raycast_frames(ego, rect, flags, None, 50.0, 360.0, R, device=dev, out=res)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ms = float(np.mean(ts))
    tests = F * R * 4 * O
    # executed work: the instrumented twin of the kernel (fo_visibility_stats) counts what survives the culls
    cnt = torch.zeros(4, dtype=torch.int64, device=dev)
    raycast_frames(ego, rect, flags, None, 50.0, 360.0, R, device=dev, out=res, stats=cnt)
    torch.cuda.synchronize()
    exec_tests, skipped, staged, listed = (float(v) for v in cnt.cpu().tolist())
    # instruction model of the cast: ~18 issue slots per executed test (2 LDS.128/64, 6 FP32, 4 compares, vote, loop),
    # ~5 per skipped (warp, edge) pair; 10 flop per executed test
    out["visibility"] = {"workload": "C-vis 10000 frames x 4096 rays x 512 rectangles", "kernel_ms": ms,
                         "frames_per_s": F / (ms * 1e-3), "ray_edge_tests_per_s": tests / (ms * 1e-3),
                         "roofline": {"bound": "fp32", "kernel": "fo_visibility_kernel", "unit": "TFLOP/s",
                                      "achieved": exec_tests * 10 / (ms * 1e-3) / 1e12, "peak": fp32_peak,
                                      "frac": exec_tests * 10 / (ms * 1e-3) / 1e12 / fp32_peak, "peak_source": fp32_src,
                                      "executed_tests_per_frame": exec_tests / F, "brute_force_tests_per_frame": tests / F,
                                      "skipped_warp_edge_pairs_per_frame": skipped / F, "staged_edges_per_frame": staged / F,
                                      "fan_list_entries_per_frame": listed / F,
                                      "effective_achieved": tests * 20 / (ms * 1e-3) / 1e12,
                                      "effective_frac": tests * 20 / (ms * 1e-3) / 1e12 / fp32_peak,
                                      "note": "frac: ray x edge tests the kernel really executes (counted by its instrumented "
                                              "twin, fo_visibility_stats: after the sensor-disc cull, the per-fan sector cull and "
                                              "the near-to-far skip of edges beyond the warp's farthest hit), 10 flop each; "
                                              "effective_frac: SURVEY.md 8d's algorithmic 20 flop per brute-force ray x edge test "
                                              "-- it measures the culling, not the pipes.  The kernel is issue-bound, not "
                                              "FP32-bound (profiles/ncu_r2_visibility_summary.txt)",
                                      "hbm_frac": F * (O * 21 + R * 8 + O) / (ms * 1e-3) / 1e9 / hbm_peak,
                                      "algorithmic_bytes": F * (O * 21 + R * 8 + O)}}
    # the same frames with a 400-segment road-border ring (real scenes always have one: 350-400 border edges)
    try:
        ring = np.stack([np.array([45.0 * np.cos(a0), 45.0 * np.sin(a0), 45.0 * np.cos(a1), 45.0 * np.sin(a1)], dtype=np.float32)
                         for a0, a1 in zip(np.linspace(0, 2 * np.pi, 401)[:-1], np.linspace(0, 2 * np.pi, 401)[1:])])
        ring_d = torch.from_numpy(ring).to(dev)
        res = raycast_frames(ego, rect, flags, ring_d, 50.0, 360.0, R, device=dev, out=res)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            raycast_frames(ego, rect, flags, ring_d, 50.0, 360.0, R, device=dev, out=res)
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        out["visibility"]["with_400_segment_border_ring_ms"] = float(np.mean(ts))
    except Exception as e:
        out["visibility"]["with_400_segment_border_ring_ms"] = repr(e)
    del rect, flags, ego, res
    # ---- detail-output variant of the dense core (per-pair and per-step arrays materialised; SURVEY.md 8d) ---------
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    nd, ad, td = 20000, 64, 51
    case = S.make_case(nd, ad, td)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"], device=str(dev))
    eng.set_agents(AgentSet.from_case(case["agents"]))
    ego_d = torch.from_numpy(case["ego"].astype(np.float32)).to(dev)
    r = eng.assess(ego_d, want_pair=True, want_step=True)
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.assess(ego_d, want_pair=True, want_step=True, out=r)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ms = float(np.median(ts))
    wr = (r.pair.numel() + r.step.numel()) * 4
    rd = nd * td * 20 + ad * td * 44
    out["detail_kernel"] = {"workload": f"{nd} trajectories x {ad} agents x {td - 1} steps, pair[N,A,12] and step[N,A,T-1,3] written",
                            "kernel_ms": ms, "evals_per_s": nd * ad * (td - 1) / (ms * 1e-3),
                            "written_GB_per_s": wr / (ms * 1e-3) / 1e9,
                            "roofline": {"bound": "hbm", "kernel": "fo_metric_detail_kernel", "unit": "GB/s",
                                         "achieved": (wr + rd) / (ms * 1e-3) / 1e9, "peak": hbm_peak,
                                         "frac": (wr + rd) / (ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                                         "algorithmic_bytes": wr + rd,
                                         "note": "12 B per evaluation + 48 B per pair written, bundle and agent table read "
                                                 "once; the kernel is instruction-issue bound (profiles/ncu_r2_detail_*): "
                                                 "both harm values per step, collision probability inside the gate and the "
                                                 "BE bisections cost more issue slots than the stores cost bandwidth"}}
    del r, ego_d, eng
    # ---- stage 2: constant-velocity rollout of 256 phantom agents x 51 states ----------------------------------
    rng = np.random.default_rng(5)
    x0, y0, v, phi = rng.uniform(-50, 50, 256), rng.uniform(-50, 50, 256), rng.uniform(1, 10, 256), rng.uniform(-3, 3, 256)
    rollout_cv(x0, y0, v, phi, 0.1, 5.0, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        rollout_cv(x0, y0, v, phi, 0.1, 5.0, device=dev)
    torch.cuda.synchronize()
    out["rollout_cv"] = {"workload": "256 agents x 51 states, host arrays in, device table out",
                         "wall_us_per_call": (time.perf_counter() - t0) / 20 * 1e6}
    # ---- one whole planning cycle on the reference's scenario1 (compact scene fixture) ---------------------------
    scene = os.path.join(ROOT, "tests", "golden", "scene_scenario1.json")
    if os.path.exists(scene):
        from frenetix_occlusion_b200 import replay as RP
        from frenetix_occlusion_b200.interface import FOInterface
        from frenetix_occlusion_b200.scenario import scenario_from_dict
        with open(scene) as f:
            doc = json.load(f)
        random.seed(7)
        sc = scenario_from_dict(doc["scene"])
        eg = RP.OpenLoopEgo(sc)
        fo = FOInterface(sc, eg.reference_path, RP.DEFAULT_VEHICLE, sc.dt, config_path=RP.deployment_config(), device=str(dev))
        t_eval, t_assess, n_sp = [], [], []
        per_traj_us = per_traj_prefetched_us = None
        for ts_ in (0, 6, 12, 18):
            st = eg.state(ts_)
            fan = torch.from_numpy(RP.frenet_fan(eg.cosy, st["pos_cl"][0], st["pos_cl"][1], st["v"],
                                                 speed_factors=np.linspace(0, 1.3, 40), lateral_targets=np.linspace(-1.5, 1.5, 25)
                                                 ).astype(np.float32)).to(dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fo.evaluate_scenario({}, st["pos"], st["orientation"], st["pos_cl"], st["v"], ts_, eg.cosy)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            r = fo.assess_bundle(fan)
            nvalid = int(r.valid.sum().item())
            t2 = time.perf_counter()
            if ts_ == 6 and fo.agent_manager.predictions:
                # the reference's per-trajectory protocol: one call per candidate (interface.py:216-219)
                host_fan = fan[:40].cpu().numpy().astype(np.float64)
                trajs = []
                for q in range(len(host_fan)):
                    tr = type("T", (), {})()
                    tr.cartesian = type("C", (), {})()
                    tr.cartesian.x, tr.cartesian.y, tr.cartesian.theta, tr.cartesian.v, tr.cartesian.a = \
                        (host_fan[q, :, c] for c in range(5))
                    trajs.append(tr)
                fo.trajectory_safety_assessment(trajs[0])
                tq = time.perf_counter()
                for tr in trajs[1:]:
                    fo.trajectory_safety_assessment(tr)
                per_traj_us = (time.perf_counter() - tq) / (len(trajs) - 1) * 1e6
                # the same protocol after handing the candidate list over once: one launch, answers from the host copy
                tq = time.perf_counter()
                fo.prefetch_assessments(trajs)
                for tr in trajs:
                    fo.trajectory_safety_assessment(tr)
                per_traj_prefetched_us = (time.perf_counter() - tq) / len(trajs) * 1e6
            t_eval.append((t1 - t0) * 1e3)
            t_assess.append((t2 - t1) * 1e3)
            n_sp.append((len(fo.spawn_points), len(fo.agent_manager.predictions), nvalid))
        out["planning_cycle"] = {"workload": "scenario1 (left turn, truck-occluded cyclist), 1000-trajectory fan, default metrics",
                                 "evaluate_scenario_ms": t_eval, "assess_bundle_ms": t_assess,
                                 "spawn_points_predictions_valid": n_sp,
                                 "trajectory_safety_assessment_us_per_call": per_traj_us,
                                 "trajectory_safety_assessment_prefetched_us_per_call": per_traj_prefetched_us,
                                 "note": "host wall clock; evaluate_scenario = visibility + spawn locator (host bookkeeping on "
                                         "GPU-classified samples) + rollouts; assess_bundle = pack + one kernel + read-back"}
    return out


_REAL_STDOUT = None


def _quiet_stdout():
    """Libraries under us print to the C-level stdout (NCCL's version banner): keep stdout for the ONE JSON line by
    pointing fd 1 at stderr for the duration of the run and writing the line to the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def _emit(line: dict):
    text = json.dumps(line) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, text.encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c-sweep", choices=["c-sweep", "c-lat"])
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: result exchange fused into the kernel (peer-mapped buffers) or NCCL all-gather")
    ap.add_argument("--e2e-torch", action="store_true", help="N > 1: time the e2e step on the torch path instead of the C-ABI host call")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-stages", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result arrays of the last timed step as DIR/<name>.npy (same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
