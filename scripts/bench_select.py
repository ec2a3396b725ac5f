"""First valid row per problem (fo_metric_batch_select) against the full batch call followed by a device argmax and a
one-int read-back; prints one JSON line.

A planner sorts its candidates by cost and takes the first one that passes.  Both paths give it that index on the host:
  select  MetricEngine.select / select_batch, then selected.cpu();
  full    MetricEngine.assess / assess_batch, then the first valid row per problem on the device, then .cpu().
Bundles are device-resident and already in each problem's frame, so neither path pays a host staging.  The two paths
alternate, twice, on the same card; median and range are reported, with the rows the select call assessed
(valid != FO_VALID_SKIPPED).  Every run checks that selected equals the first valid row of the full call.

Workloads (seeded; thresholds armed with harm 0.1 so that enough rows fail to place the first valid one):
  clat-diag / clat-corr    one problem, 1000 x 32 agents x T = 31, diagonal / correlated covariances;
  fleet-diag / fleet-corr  the fleet of bench_batch_corr.py: 256 problems x 1000 x 31, 1..8 agents, all diagonal / all
                           correlated;
  big-diag / big-corr      one problem, 1 M x 256 agents x T = 51.
Each runs with the first valid row at rank 0, at N/2 and with none valid ("none"), got by reordering the rows of the
case after one full pass (invalid rows repeat where there are too few).

    python scripts/bench_select.py [--steps 10] [--warmup 2] [--workloads clat-diag,clat-corr,fleet-diag,fleet-corr]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_batch import gpu_info  # noqa: E402
from bench_batch_corr import correlate  # noqa: E402
from bench_batch_vehicles import fleet  # noqa: E402

THRESHOLDS = {"harm": 0.1, "risk": None, "be": None, "cp": None, "ttc": None, "wttc": None, "ttce": None, "dce": None}
# tried in order until a case's full pass has valid and invalid rows: harm 0.1; then risk and CP armed as well; then the
# same with the agents pulled onto the ego paths (positions x 0.3).  None of them arms a rounding-tie clause.
ARMINGS = ((THRESHOLDS, 1.0), ({**THRESHOLDS, "risk": 0.01, "cp": 0.05}, 1.0), ({**THRESHOLDS, "risk": 0.01, "cp": 0.05}, 0.3))
POSITIONS = ("0", "N/2", "none")


def reorder(valid, pos):
    """Row order with the first valid row at rank pos (0 / N/2) or none valid.  A problem without invalid rows keeps its
    order (first valid row 0), one without valid rows too (none valid)."""
    N = len(valid)
    good, bad = np.flatnonzero(valid == 1), np.flatnonzero(valid != 1)
    if len(bad) == 0 or len(good) == 0:
        return np.arange(N)
    if pos == "none":
        return np.resize(bad, N)
    k = 0 if pos == "0" else N // 2
    return np.concatenate([np.resize(bad, k), good[:1], np.arange(N)[:N - k - 1]])


def first_valid(valid, n):
    """First valid row of each of the equal-sized problems of a flat valid tensor (n when none), on the device."""
    import torch
    v = (valid.view(-1, n) == 1)
    return torch.where(v.any(1), v.to(torch.int32).argmax(1), torch.full_like(v[:, 0], n, dtype=torch.int64))


def make_problems(wl, arming):
    import corr_oracle as CO
    from bench_batch import problems
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    if wl.startswith("fleet"):
        probs, case = problems(256, 1000, 31, lambda r: r.integers(1, 9), seed=1)
        case["thresholds"] = arming[0]
        for ag, _, _ in probs:
            ag.x, ag.y = ag.x * arming[1], ag.y * arming[1]
        rng = np.random.default_rng(11)
        if wl == "fleet-corr":
            probs = [(correlate(ag, rng), o, e) for ag, o, e in probs]
        return probs, case, fleet(256, 1)
    n, a, t = (1000, 32, 31) if wl.startswith("clat") else (1_000_000, 256, 51)
    case = S.make_case(n, a, t, seed=7, thresholds=arming[0])
    for ag in case["agents"]:
        ag["pos"] = np.asarray(ag["pos"]) * arming[1]
    if wl.endswith("corr"):
        case = CO.add_correlations(case, 7)
    ag = AgentSet.from_case(case["agents"])
    return [(ag, (float(ag.x[0, 0]), float(ag.y[0, 0])), case["ego"])], case, None


def bench(wl, steps, warmup):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import MetricEngine
    for arming in ARMINGS:
        probs, case, vehicles = make_problems(wl, arming)
        single = vehicles is None
        eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
        dev = [torch.from_numpy((e - np.array([o[0], o[1], 0, 0, 0])).astype(np.float32)).cuda() for _, o, e in probs]
        if single:
            eng.set_agents(probs[0][0])
            full_call = lambda d: eng.assess(d[0])                # noqa: E731
            sel_call = lambda d: eng.select(d[0])                 # noqa: E731
        else:
            eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=vehicles, correlated=True)
            eng._batch["origins"] = np.zeros_like(eng._batch["origins"])
            full_call = lambda d: eng.assess_batch(d)             # noqa: E731
            sel_call = lambda d: eng.select_batch(d)              # noqa: E731
        n = int(dev[0].shape[0])
        valid0 = [v.cpu().numpy() for v in full_call(dev).valid.view(len(dev), n)]
        frac = float(np.mean(np.concatenate(valid0)))
        if 0.0 < frac < 0.9:
            break
    out = []
    for pos in POSITIONS:
        d = [x[torch.from_numpy(reorder(v, pos)).cuda()].contiguous() for x, v in zip(dev, valid0)]
        full_idx = lambda: first_valid(full_call(d).valid, n).cpu()   # noqa: E731
        sel_idx = lambda: sel_call(d).selected.cpu()                  # noqa: E731

        def host_time(fn):
            for _ in range(warmup):
                fn()
            ts = []
            for _ in range(steps):
                t0 = time.perf_counter()
                fn()
                ts.append((time.perf_counter() - t0) * 1e3)
            return ts
        t_sel, t_full = [], []
        for _ in range(2):                         # alternate the two paths, twice
            t_sel += host_time(sel_idx)
            t_full += host_time(full_idx)
        r = sel_call(d)
        want = first_valid(full_call(d).valid, n).cpu().numpy()
        got = r.selected.cpu().numpy()
        assessed = int((r.valid != L.FO_VALID_SKIPPED).sum().item())
        med = lambda x: float(np.median(x))       # noqa: E731
        rng_ = lambda x: [float(min(x)), float(max(x))]   # noqa: E731
        out.append({"workload": wl, "first_valid": pos, "P": len(dev), "N_total": n * len(dev),
                    "A": [int(p[0].n_agents) for p in probs][:1] if single else "1..8", "T": int(dev[0].shape[1]),
                    "thresholds": {k: v for k, v in arming[0].items() if v is not None}, "agent_scale": arming[1],
                    "valid_fraction": frac,
                    "select_ms": med(t_sel), "select_ms_range": rng_(t_sel),
                    "full_ms": med(t_full), "full_ms_range": rng_(t_full), "speedup": med(t_full) / med(t_sel),
                    "rows_assessed": assessed, "selected_equal": bool(np.array_equal(got, want))})
        del d
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="clat-diag,clat-corr,fleet-diag,fleet-corr,big-diag,big-corr")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_select.py needs a CUDA device")
    res = {"gpu": gpu_info(), "results": []}
    for wl in args.workloads.split(","):
        if wl not in ("clat-diag", "clat-corr", "fleet-diag", "fleet-corr", "big-diag", "big-corr"):
            ap.error(f"unknown workload {wl}")
        res["results"] += bench(wl, args.steps, args.warmup)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
