"""Batches of independent planning problems with one ego vehicle per problem (a mixed fleet) against the per-problem loop;
prints one JSON line.

Workloads (seeded, built from synthetic.make_case like scripts/bench_batch.py; problem p's vehicle is one of four classes
-- compact, the synthetic.VEHICLE sedan, van, truck -- with its dimensions, mass and a_max jittered, so no two match):
  fleet         P = 256 problems x 1000 trajectories x T = 31, A_p drawn from 1..8, all 7 metrics.  The batch
                (set_agent_batch(..., vehicles) + assess_batch + copies of valid / flags / summary to the host) is timed
                against the loop that is the only option without per-problem vehicles (one engine per vehicle,
                set_agents + assess + the same copies, per problem), host arrays in to host copies out, with a host
                clock ending in a synchronise; the metric call alone on device-resident bundles is timed with CUDA events.
                The outputs of both paths are compared bit for bit;
  fleet-detail  the same with P = 256 x 300 x 31 and pair + step (assess_batch(want_pair, want_step)), all five outputs
                copied to the host and compared.  Run it in a process of its own (--workloads fleet-detail): after
                the fleet workload in the same process its batched host time has been measured three times lower,
                an effect of the host copies, not of the metric call.

    python scripts/bench_batch_vehicles.py [--steps 10] [--warmup 2] [--workloads fleet,fleet-detail]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_batch import gpu_info, problems  # noqa: E402

# compact, sedan (synthetic.VEHICLE), van, truck
CLASSES = ({"length": 3.6, "width": 1.6, "mass": 900.0, "wb_rear_axle": 1.1, "a_max": 9.5},
           None,
           {"length": 5.9, "width": 2.0, "mass": 2500.0, "wb_rear_axle": 1.8, "a_max": 8.0},
           {"length": 12.0, "width": 2.55, "mass": 18000.0, "wb_rear_axle": 3.9, "a_max": 6.0})


def fleet(n, seed):
    from frenetix_occlusion_b200 import synthetic as S
    rng = np.random.default_rng(seed)
    return [{k: float(np.float32(v * rng.uniform(0.96, 1.04))) for k, v in (CLASSES[p % 4] or S.VEHICLE).items()}
            for p in range(n)]


def bench_fleet_vs_loop(name, probs, case, vehicles, detail, steps, warmup):
    import torch
    from frenetix_occlusion_b200.engine import MetricEngine
    mk = lambda v: MetricEngine(v, case["dt"], case["activated_metrics"], case["thresholds"])  # noqa: E731
    eng_b = mk(case["vehicle"])
    eng_l = [mk(v) for v in vehicles]            # one engine per vehicle, as every planner of the fleet holds its own
    ags, orgs, egos = [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs]
    fields = ("valid", "flags", "summary") + (("pair", "step") if detail else ())
    host = lambda r: [getattr(r, f).cpu().numpy() for f in fields]  # noqa: E731
    sync = torch.cuda.synchronize

    def batched():
        eng_b.set_agent_batch(ags, orgs, vehicles=vehicles)
        return host(eng_b.assess_batch(egos, want_pair=detail, want_step=detail))

    def loop():
        out = []
        for eng, ag, o, e in zip(eng_l, ags, orgs, egos):
            eng.set_agents(ag, origin=o)
            out.append(host(eng.assess(e, want_pair=detail, want_step=detail)))
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
    # the metric call alone (CUDA events): assess_batch on device-resident bundles already in each problem's frame
    eng_b.set_agent_batch(ags, orgs, vehicles=vehicles)
    dev = [torch.from_numpy((e - np.array([o[0], o[1], 0, 0, 0])).astype(np.float32)).cuda() for e, o in zip(egos, orgs)]
    eng_b._batch["origins"] = np.zeros_like(eng_b._batch["origins"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        eng_b.assess_batch(dev, want_pair=detail, want_step=detail)
    t_metric = []
    for _ in range(steps):
        e0.record()
        eng_b.assess_batch(dev, want_pair=detail, want_step=detail)
        e1.record()
        sync()
        t_metric.append(e0.elapsed_time(e1))
    eng_b.set_agent_batch(ags, orgs, vehicles=vehicles)
    parts = eng_b.assess_batch(egos, want_pair=detail, want_step=detail).split()
    res_l = loop()
    equal = all(np.array_equal(g, w, equal_nan=True) and g.shape == w.shape
                for gp, wp in zip(parts, res_l) for g, w in zip(host(gp), wp))
    med = lambda x: float(np.median(x))  # noqa: E731
    return {"workload": name, "P": len(probs), "N_total": sum(len(e) for e in egos), "T": int(egos[0].shape[1]),
            "detail": detail, "distinct_vehicles": len({tuple(v.values()) for v in vehicles}),
            "agents": [int(a.n_agents) for a in ags][:8] + (["..."] if len(ags) > 8 else []),
            "batched_ms": med(t_batch), "batched_ms_range": [min(t_batch), max(t_batch)],
            "loop_ms": med(t_loop), "loop_ms_range": [min(t_loop), max(t_loop)],
            "speedup": med(t_loop) / med(t_batch), "metric_call_ms": med(t_metric),
            "metric_call_ms_range": [min(t_metric), max(t_metric)], "outputs_equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="fleet,fleet-detail")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_batch_vehicles.py needs a CUDA device")
    res = {"gpu": gpu_info(), "results": []}
    for wl in args.workloads.split(","):
        if wl == "fleet":
            probs, case = problems(256, 1000, 31, lambda r: r.integers(1, 9), seed=1)
            res["results"].append(bench_fleet_vs_loop(wl, probs, case, fleet(256, 1), False, args.steps, args.warmup))
        elif wl == "fleet-detail":
            probs, case = problems(256, 300, 31, lambda r: r.integers(1, 9), seed=3)
            res["results"].append(bench_fleet_vs_loop(wl, probs, case, fleet(256, 3), True, args.steps, args.warmup))
        else:
            ap.error(f"unknown workload {wl}")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
