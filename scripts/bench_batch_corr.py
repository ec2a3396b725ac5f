"""Batches with correlated prediction covariances (set_agent_batch(..., correlated=True): fo_agents_pack_batch_corr +
fo_metric_batch[_detail]_corr) against the per-problem loop; prints one JSON line.

Workloads (seeded, the fleets of scripts/bench_batch_vehicles.py: problem p has its own jittered vehicle; a correlated
problem's covariances get var_x, var_y scaled by U(0.5, 2) each and rho ~ U(-0.9, 0.9) per state, float32 values):
  fleet-corr         P = 256 problems x 1000 trajectories x T = 31, A_p drawn from 1..8, all 7 metrics, every problem
                     correlated;
  fleet-mixed        the same with every second problem correlated (the others diagonal);
  fleet-corr-detail  P = 256 x 300 x 31, every problem correlated, pair + step.
Each is timed end to end (host arrays in, host copies of every output out, host clock ending in a synchronise) against
the loop that is the only option without correlated batches: one engine per vehicle, set_agents + assess + the same
copies, per problem.  The two paths alternate, twice; the median and range are reported.  The metric call alone on
device-resident bundles is timed with CUDA events.  The outputs of both paths are compared bit for bit.

    python scripts/bench_batch_corr.py [--steps 10] [--warmup 2] [--workloads fleet-corr,fleet-mixed,fleet-corr-detail]
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
from bench_batch_vehicles import fleet  # noqa: E402


def correlate(ag, rng):
    """Correlated covariances of the same agents (positive definite on every state)."""
    f32 = lambda z: z.astype(np.float32).astype(np.float64)  # noqa: E731
    ag.var_x = f32(ag.var_x * rng.uniform(0.5, 2.0, ag.var_x.shape))
    ag.var_y = f32(ag.var_y * rng.uniform(0.5, 2.0, ag.var_y.shape))
    ag.cov_xy = f32(rng.uniform(-0.9, 0.9, ag.var_x.shape) * np.sqrt(ag.var_x * ag.var_y))
    return ag


def bench(name, probs, case, vehicles, detail, steps, warmup):
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
        eng_b.set_agent_batch(ags, orgs, vehicles=vehicles, correlated=True)
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

    # the metric call alone (CUDA events) on device-resident bundles already in each problem's frame: the batch call,
    # and the loop's metric calls (tables packed beforehand)
    dev = [torch.from_numpy((e - np.array([o[0], o[1], 0, 0, 0])).astype(np.float32)).cuda() for e, o in zip(egos, orgs)]
    eng_b.set_agent_batch(ags, orgs, vehicles=vehicles, correlated=True)
    eng_b._batch["origins"] = np.zeros_like(eng_b._batch["origins"])
    for eng, ag in zip(eng_l, ags):
        eng.set_agents(ag)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def ev_time(fn):
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(steps):
            e0.record()
            fn()
            e1.record()
            sync()
            ts.append(e0.elapsed_time(e1))
        return ts
    m_batch, m_loop = [], []
    for _ in range(2):
        m_batch += ev_time(lambda: eng_b.assess_batch(dev, want_pair=detail, want_step=detail))
        m_loop += ev_time(lambda: [eng.assess(d, want_pair=detail, want_step=detail) for eng, d in zip(eng_l, dev)])

    eng_b.set_agent_batch(ags, orgs, vehicles=vehicles, correlated=True)
    parts = eng_b.assess_batch(egos, want_pair=detail, want_step=detail).split()
    res_l = loop()
    equal = all(np.array_equal(g, w, equal_nan=True) and g.shape == w.shape
                for gp, wp in zip(parts, res_l) for g, w in zip(host(gp), wp))
    med = lambda x: float(np.median(x))  # noqa: E731
    rng_ = lambda x: [float(min(x)), float(max(x))]  # noqa: E731
    return {"workload": name, "P": len(probs), "N_total": sum(len(e) for e in egos), "T": int(egos[0].shape[1]),
            "detail": detail, "correlated_problems": sum(a.cov_xy is not None for a in ags),
            "batched_ms": med(t_batch), "batched_ms_range": rng_(t_batch),
            "loop_ms": med(t_loop), "loop_ms_range": rng_(t_loop), "speedup": med(t_loop) / med(t_batch),
            "metric_call_ms": med(m_batch), "metric_call_ms_range": rng_(m_batch),
            "loop_metric_calls_ms": med(m_loop), "loop_metric_calls_ms_range": rng_(m_loop),
            "outputs_equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="fleet-corr,fleet-mixed,fleet-corr-detail")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_batch_corr.py needs a CUDA device")
    res = {"gpu": gpu_info(), "results": []}
    for wl in args.workloads.split(","):
        if wl in ("fleet-corr", "fleet-mixed"):
            probs, case = problems(256, 1000, 31, lambda r: r.integers(1, 9), seed=1)
            every, vehicles, detail = (1 if wl == "fleet-corr" else 2), fleet(256, 1), False
        elif wl == "fleet-corr-detail":
            probs, case = problems(256, 300, 31, lambda r: r.integers(1, 9), seed=3)
            every, vehicles, detail = 1, fleet(256, 3), True
        else:
            ap.error(f"unknown workload {wl}")
        rng = np.random.default_rng(11)
        probs = [((correlate(ag, rng) if p % every == 0 else ag), o, e) for p, (ag, o, e) in enumerate(probs)]
        res["results"].append(bench(wl, probs, case, vehicles, detail, args.steps, args.warmup))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
