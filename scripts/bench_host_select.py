"""First valid row per problem from host memory (fo_metric_batch_host_select) against fo_metric_batch_host_corr followed
by a host scan of valid for each problem's first valid row; prints one JSON line.

Both paths take the same host arrays (float64 ego rows in the world frame, one origin per problem, the agents and their
covariances) and give the planner its index on the host.  The host call copies every row across PCIe and assesses every
row; the select call assesses rank windows in rounds and copies only the rows of those windows (DESIGN.md 5.15).

Workloads (seeded): the fleet of bench_batch_corr.py, 256 problems x 1000 x 31, 1..8 agents, one vehicle each, all
diagonal ("fleet-diag") or all correlated ("fleet-corr"), thresholds armed as in bench_select.py.  Each runs with
pageable (numpy) and page-locked (torch pin_memory) rows, and with the first valid row at rank 0, at N/2 and with none
valid, got by reordering the rows after one full pass.  The two paths alternate, twice; median and range of host-clock
times (each call ends in a synchronise) are reported, with the rows the select call assessed (valid !=
FO_VALID_SKIPPED), the rows it copied and its rounds (from the window rule and the selections).  Every run checks that
the selections are equal.

    python scripts/bench_host_select.py [--steps 10] [--warmup 2] [--workloads fleet-diag,fleet-corr]
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

from bench_batch import gpu_info, team_warps  # noqa: E402
from bench_select import ARMINGS, POSITIONS, make_problems, reorder  # noqa: E402


def windows(selected, n, w0):
    """Rows copied and rounds of the window rule for problems of n rows with these selections."""
    copied, rounds = 0, 0
    for s in selected:
        start, length, r = 0, w0, 0
        while True:
            take = min(length, n - start)
            copied, r = copied + take, r + 1
            if s < start + take or start + take == n:
                break
            start, length = start + take, 4 * length
        rounds = max(rounds, r)
    return copied, rounds


def bench(wl, steps, warmup):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import MetricEngine
    from test_metric_batch_host import _params
    from test_metric_batch_host_select import _full, _inputs, _select
    for arming in ARMINGS:
        probs, case, vehicles = make_problems(wl, arming)
        eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
        params = _params(eng)
        ags, orgs, egos = [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs]
        x = _inputs(L, ags, orgs, egos, vehicles)
        n = len(egos[0])
        valid0 = _full(L, params, x)["valid"].reshape(len(egos), n)
        if 0.0 < float(valid0.mean()) < 0.9:
            break
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    a_min = min(a.n_agents for a in ags)
    teams = sms * 8 * 4 // team_warps(len(egos) * n, 31, a_min, sms)
    w0 = max(32, -(-teams // len(egos)))
    out = []
    for pinned in (False, True):
        for pos in POSITIONS:
            x = _inputs(L, ags, orgs, [e[reorder(v, pos)] for e, v in zip(egos, valid0)], vehicles, pinned=pinned)
            P = x["P"]

            def sel_idx():
                rc, r = _select(L, params, x)
                L.check(rc, "fo_metric_batch_host_select")
                return r

            def full_idx():
                v = _full(L, params, x)["valid"].reshape(P, n) == 1
                return np.where(v.any(1), v.argmax(1), n)

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
            r = sel_idx()
            want = full_idx()
            assert np.array_equal(r["selected"], want), (wl, pos, pinned)
            copied, rounds = windows(r["selected"], n, w0)
            med = lambda t: float(np.median(t))  # noqa: E731
            rng_ = lambda t: [float(min(t)), float(max(t))]  # noqa: E731
            out.append({"workload": wl, "rows": "page-locked" if pinned else "pageable", "first_valid": pos,
                        "P": P, "N_total": x["N"], "T": x["T"], "w0": w0,
                        "select_ms": med(t_sel), "select_ms_range": rng_(t_sel),
                        "host_call_scan_ms": med(t_full), "host_call_scan_ms_range": rng_(t_full),
                        "speedup": med(t_full) / med(t_sel),
                        "rows_assessed": int((r["valid"] != L.FO_VALID_SKIPPED).sum()), "rows_copied": copied,
                        "rounds": rounds, "selected_equal": True})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="fleet-diag,fleet-corr")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_host_select.py needs a CUDA device")
    res = {"gpu": gpu_info(), "results": []}
    for wl in args.workloads.split(","):
        if wl not in ("fleet-diag", "fleet-corr"):
            ap.error(f"unknown workload {wl}")
        res["results"] += bench(wl, args.steps, args.warmup)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
