"""Batches of independent planning problems against the per-problem loop; prints one JSON line.

Workloads (seeded, built from synthetic.make_case):
  multi-ego    P = 256 problems x 1000 trajectories x T = 31, A_p drawn from 1..8, all 7 metrics -- one planner per
               vehicle of a multi-agent simulation, the case the batch exists for (small problems, launch-bound loop);
  large-agent  P = 64 x 1000 x T = 51 x A_p = 32 -- the batch's one-warp window-filter class;
  c-sweep-p1   one problem of 1 M x 256 x 51 through fo_metric_batch and through fo_metric_bundle, alternating in one
               process: what the batch adds per trajectory (problem lookup, per-problem table pointers).
For the first two the batched path (set_agent_batch + assess_batch, host arrays in, host clock ending in a synchronise;
and the metric call alone on device-resident bundles, CUDA events) is timed against the loop the batch replaces
(set_agents + assess per problem, host clock ending in a synchronise).  Outputs of both are compared bit for bit, the
loop run for that comparison under FO_TEAM_WARPS set to the batch's team size.

    python scripts/bench_batch.py [--steps 10] [--warmup 2] [--workloads multi-ego,large-agent,c-sweep-p1]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as e:                      # reported, not guessed
        info["power_limit_w"] = None
        info["power_limit_error"] = repr(e)
    return info


def problems(n_problems, n_traj, n_states, agents, seed):
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    rng = np.random.default_rng(seed)
    out = []
    for p in range(n_problems):
        A = int(agents(rng))
        case = S.make_case(n_traj, A, n_states, seed=seed * 10000 + p)
        ag = AgentSet.from_case(case["agents"])
        origin = (float(ag.x[0, 0]), float(ag.y[0, 0])) if ag.n_agents else (0.0, 0.0)
        out.append((ag, origin, case["ego"]))
    return out, case


def team_warps(n_traj, n_states, a_min, sms):
    """The batch's team size as fo_metric_batch picks it (pick_team_warps in fo_metric_sweep.cu)."""
    lg = next(l for l in range(6) if (1 << l) >= a_min or l == 5)
    return max(1, min(sms * 8 * 4 // max(n_traj, 1), n_states // (4 * (32 >> lg)), 8))


def bench_batch_vs_loop(name, probs, case, steps, warmup, sms):
    import torch
    from frenetix_occlusion_b200.engine import MetricEngine
    mk = lambda: MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])  # noqa: E731
    eng_b, eng_l = mk(), mk()
    ags, orgs, egos = [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs]
    sync = torch.cuda.synchronize

    def batched():
        eng_b.set_agent_batch(ags, orgs)
        return eng_b.assess_batch(egos)

    def loop():
        out = []
        for ag, o, e in zip(ags, orgs, egos):
            eng_l.set_agents(ag, origin=o)
            out.append(eng_l.assess(e))
        return out

    def host_time(fn):
        for _ in range(warmup):
            fn()
        sync()
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            fn()
            sync()
            ts.append((time.perf_counter() - t0) * 1e3)
        return ts

    t_batch, t_loop = [], []
    for _ in range(2):                         # alternate the two paths, twice
        t_batch += host_time(batched)
        t_loop += host_time(loop)
    # metric call alone (CUDA events): assess_batch on device-resident bundles already in each problem's frame, so
    # the timed region is their concatenation on the device and the fo_metric_batch call
    eng_b.set_agent_batch(ags, orgs)
    dev = [torch.from_numpy((e - np.array([o[0], o[1], 0, 0, 0])).astype(np.float32)).cuda() for e, o in zip(egos, orgs)]
    eng_b._batch["origins"] = np.zeros_like(eng_b._batch["origins"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        eng_b.assess_batch(dev)
    t_metric = []
    for _ in range(steps):
        e0.record()
        eng_b.assess_batch(dev)
        e1.record()
        sync()
        t_metric.append(e0.elapsed_time(e1))
    # outputs: batch vs the loop under the batch's team size
    N = sum(len(e) for e in egos)
    W = team_warps(N, egos[0].shape[1], min(a.n_agents for a in ags), sms)
    res_b = batched()
    os.environ["FO_TEAM_WARPS"] = str(W)
    res_l = loop()
    sync()
    del os.environ["FO_TEAM_WARPS"]
    equal = all(np.array_equal(getattr(g, f).cpu().numpy(), getattr(w, f).cpu().numpy(), equal_nan=True)
                for g, w in zip(res_b.split(), res_l) for f in ("valid", "flags", "summary"))
    med = lambda x: float(np.median(x))  # noqa: E731
    return {"workload": name, "P": len(probs), "N_total": N, "T": int(egos[0].shape[1]),
            "agents": [int(a.n_agents) for a in ags][:8] + (["..."] if len(ags) > 8 else []),
            "team_warps": W, "batched_ms": med(t_batch), "batched_ms_range": [min(t_batch), max(t_batch)],
            "loop_ms": med(t_loop), "loop_ms_range": [min(t_loop), max(t_loop)],
            "speedup": med(t_loop) / med(t_batch), "metric_only_ms": med(t_metric),
            "metric_only_ms_range": [min(t_metric), max(t_metric)], "outputs_equal": bool(equal)}


def bench_sweep_p1(steps, warmup):
    """fo_metric_batch with P = 1 against fo_metric_bundle on the C-sweep shape, alternating, CUDA events."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet, BundleResult, MetricEngine
    N, A, T = 1_000_000, 256, 51
    case = S.make_case(1, A, T)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    chunks = [torch.from_numpy(S.ego_bundle(min(100_000, N - lo), T, seed=S.SEED + 100 + k).astype(np.float32))
              for k, lo in enumerate(range(0, N, 100_000))]
    ego = torch.cat(chunks).cuda()
    out = [BundleResult(torch.empty(N, dtype=torch.uint8, device="cuda"),
                        torch.empty((N, L.FO_SUMMARY_K), dtype=torch.float32, device="cuda"),
                        torch.empty(N, dtype=torch.int32, device="cuda")) for _ in range(2)]
    a_bundle = eng._args(ego, out[0])
    prob = (L.FoBatchProblem * 1)()
    prob[0].traj_begin, prob[0].n_traj, prob[0].n_agents, prob[0].t_stride, prob[0].table_offset = 0, N, A, T, 0
    b = L.FoMetricBatchArgs()
    b.common = eng._args(ego, out[1])
    b.n_problems, b.problems, b.arena_bytes = 1, prob, eng._table.numel()
    st = eng._stream()
    run = {"bundle": lambda: L.check(L.lib.fo_metric_bundle(C.byref(a_bundle), st)),
           "batch": lambda: L.check(L.lib.fo_metric_batch(C.byref(b), st))}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {"bundle": [], "batch": []}
    for i in range(2 * (warmup + steps)):
        k = ("bundle", "batch")[i % 2]
        e0.record()
        run[k]()
        e1.record()
        torch.cuda.synchronize()
        if i >= 2 * warmup:
            times[k].append(e0.elapsed_time(e1))
    equal = all(np.array_equal(getattr(out[0], f).cpu().numpy(), getattr(out[1], f).cpu().numpy(), equal_nan=True)
                for f in ("valid", "flags", "summary"))
    med = {k: float(np.median(v)) for k, v in times.items()}
    return {"workload": "c-sweep-p1", "N": N, "A": A, "T": T, "steps_each": steps,
            "bundle_ms": med["bundle"], "bundle_ms_range": [min(times["bundle"]), max(times["bundle"])],
            "batch_ms": med["batch"], "batch_ms_range": [min(times["batch"]), max(times["batch"])],
            "batch_over_bundle": med["batch"] / med["bundle"], "outputs_equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="multi-ego,large-agent,c-sweep-p1")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_batch.py needs a CUDA device")
    info = gpu_info()
    res = {"gpu": info, "results": []}
    for wl in args.workloads.split(","):
        if wl == "multi-ego":
            probs, case = problems(256, 1000, 31, lambda r: r.integers(1, 9), seed=1)
            res["results"].append(bench_batch_vs_loop(wl, probs, case, args.steps, args.warmup, info["sms"]))
        elif wl == "large-agent":
            probs, case = problems(64, 1000, 51, lambda r: 32, seed=2)
            res["results"].append(bench_batch_vs_loop(wl, probs, case, args.steps, args.warmup, info["sms"]))
        elif wl == "c-sweep-p1":
            res["results"].append(bench_sweep_p1(args.steps, args.warmup))
        else:
            ap.error(f"unknown workload {wl}")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
