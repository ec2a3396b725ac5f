"""Batches of independent planning problems with per-pair and per-step detail against the per-problem loop; prints one
JSON line.

Workloads (seeded, built from synthetic.make_case like scripts/bench_batch.py):
  multi-ego-detail  P = 256 problems x 300 trajectories x T = 31, A_p drawn from 1..8, all 7 metrics, pair + step -- the
                    reference's per-trajectory protocol (prefetch_assessments) for every vehicle of a multi-agent
                    simulation.  The batched path (set_agent_batch + assess_batch(want_pair, want_step) + copies of the
                    five outputs to the host) is timed against the loop it replaces (set_agents + assess(want_pair,
                    want_step) + the same copies, per problem), host arrays in to host copies out, with a host clock
                    ending in a synchronise; the detail call alone on device-resident bundles is timed with CUDA events.
                    All five outputs of both paths are compared bit for bit;
  c-detail-p1       one problem of 20 000 x 64 x 51 (the scripts/bench_detail.py size) through fo_metric_batch_detail
                    and through fo_metric_bundle with pair + step, alternating in one process, CUDA events: what the
                    batch adds per trajectory (problem lookup, per-problem table and output pointers).

    python scripts/bench_batch_detail.py [--steps 10] [--warmup 2] [--workloads multi-ego-detail,c-detail-p1]
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
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_batch import gpu_info, problems  # noqa: E402

FIELDS = ("valid", "flags", "summary", "pair", "step")


def _host(r):
    return [getattr(r, f).cpu().numpy() for f in FIELDS]


def bench_detail_batch_vs_loop(name, probs, case, steps, warmup):
    import torch
    from frenetix_occlusion_b200.engine import MetricEngine
    mk = lambda: MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])  # noqa: E731
    eng_b, eng_l = mk(), mk()
    ags, orgs, egos = [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs]
    sync = torch.cuda.synchronize

    def batched():
        eng_b.set_agent_batch(ags, orgs)
        return _host(eng_b.assess_batch(egos, want_pair=True, want_step=True))

    def loop():
        out = []
        for ag, o, e in zip(ags, orgs, egos):
            eng_l.set_agents(ag, origin=o)
            out.append(_host(eng_l.assess(e, want_pair=True, want_step=True)))
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
    # detail call alone (CUDA events): assess_batch on device-resident bundles already in each problem's frame, so the
    # timed region is their concatenation on the device, the output allocation and the fo_metric_batch_detail call
    eng_b.set_agent_batch(ags, orgs)
    dev = [torch.from_numpy((e - np.array([o[0], o[1], 0, 0, 0])).astype(np.float32)).cuda() for e, o in zip(egos, orgs)]
    eng_b._batch["origins"] = np.zeros_like(eng_b._batch["origins"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        eng_b.assess_batch(dev, want_pair=True, want_step=True)
    t_metric = []
    for _ in range(steps):
        e0.record()
        eng_b.assess_batch(dev, want_pair=True, want_step=True)
        e1.record()
        sync()
        t_metric.append(e0.elapsed_time(e1))
    # outputs: the batch's per-problem views against the loop, all five bit for bit
    eng_b.set_agent_batch(ags, orgs)
    parts = eng_b.assess_batch(egos, want_pair=True, want_step=True).split()
    res_l = loop()
    equal = all(np.array_equal(g, w, equal_nan=True) and g.shape == w.shape
                for gp, wp in zip(parts, res_l) for g, w in zip(_host(gp), wp))
    N = sum(len(e) for e in egos)
    n_pairs = sum(len(e) * a.n_agents for e, a in zip(egos, ags))
    T = int(egos[0].shape[1])
    med = lambda x: float(np.median(x))  # noqa: E731
    return {"workload": name, "P": len(probs), "N_total": N, "T": T, "pairs": n_pairs,
            "detail_mb": n_pairs * (12 + 3 * (T - 1)) * 4 / 1e6,
            "agents": [int(a.n_agents) for a in ags][:8] + (["..."] if len(ags) > 8 else []),
            "batched_ms": med(t_batch), "batched_ms_range": [min(t_batch), max(t_batch)],
            "loop_ms": med(t_loop), "loop_ms_range": [min(t_loop), max(t_loop)],
            "speedup": med(t_loop) / med(t_batch), "detail_call_ms": med(t_metric),
            "detail_call_ms_range": [min(t_metric), max(t_metric)], "outputs_equal": bool(equal)}


def bench_detail_p1(steps, warmup):
    """fo_metric_batch_detail with P = 1 against fo_metric_bundle with pair + step, alternating, CUDA events."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet, BundleResult, MetricEngine
    N, A, T = 20_000, 64, 51
    case = S.make_case(N, A, T)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    ego = torch.from_numpy(case["ego"].astype(np.float32)).cuda()
    out = []
    for _ in range(2):
        r = BundleResult(torch.empty(N, dtype=torch.uint8, device="cuda"),
                         torch.empty((N, L.FO_SUMMARY_K), dtype=torch.float32, device="cuda"),
                         torch.empty(N, dtype=torch.int32, device="cuda"))
        r.pair = torch.empty((N, A, L.FO_PAIR_K), dtype=torch.float32, device="cuda")
        r.step = torch.empty((N, A, T - 1, L.FO_STEP_K), dtype=torch.float32, device="cuda")
        out.append(r)
    a_bundle = eng._args(ego, out[0])
    a_bundle.pair, a_bundle.step = out[0].pair.data_ptr(), out[0].step.data_ptr()
    prob = (L.FoBatchProblem * 1)()
    prob[0].traj_begin, prob[0].n_traj, prob[0].n_agents, prob[0].t_stride, prob[0].table_offset = 0, N, A, T, 0
    b = L.FoMetricBatchArgs()
    b.common = eng._args(ego, out[1])
    b.common.pair, b.common.step = out[1].pair.data_ptr(), out[1].step.data_ptr()
    b.n_problems, b.problems, b.arena_bytes = 1, prob, eng._table.numel()
    st = eng._stream()
    run = {"bundle": lambda: L.check(L.lib.fo_metric_bundle(C.byref(a_bundle), st)),
           "batch": lambda: L.check(L.lib.fo_metric_batch_detail(C.byref(b), st))}
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
                for f in FIELDS)
    med = {k: float(np.median(v)) for k, v in times.items()}
    return {"workload": "c-detail-p1", "N": N, "A": A, "T": T, "steps_each": steps,
            "bundle_ms": med["bundle"], "bundle_ms_range": [min(times["bundle"]), max(times["bundle"])],
            "batch_ms": med["batch"], "batch_ms_range": [min(times["batch"]), max(times["batch"])],
            "batch_over_bundle": med["batch"] / med["bundle"], "outputs_equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="multi-ego-detail,c-detail-p1")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_batch_detail.py needs a CUDA device")
    res = {"gpu": gpu_info(), "results": []}
    for wl in args.workloads.split(","):
        if wl == "multi-ego-detail":
            probs, case = problems(256, 300, 31, lambda r: r.integers(1, 9), seed=3)
            res["results"].append(bench_detail_batch_vs_loop(wl, probs, case, args.steps, args.warmup))
        elif wl == "c-detail-p1":
            res["results"].append(bench_detail_p1(args.steps, args.warmup))
        else:
            ap.error(f"unknown workload {wl}")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
