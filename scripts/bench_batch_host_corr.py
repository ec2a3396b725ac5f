"""A batch with correlated prediction covariances from host memory in one C-ABI call (fo_metric_batch_host_corr) against
the two ways a host caller has without it; prints one JSON line.

Workloads (seeded, those of scripts/bench_batch_corr.py: problem p has its own jittered vehicle; a correlated problem's
covariances get var_x, var_y scaled by U(0.5, 2) each and rho ~ U(-0.9, 0.9) per state, float32 values; every problem
moved by its own UTM-sized offset of 1e5-6e6 m, as in scripts/bench_batch_host.py):
  fleet-corr         P = 256 problems x 1000 trajectories x T = 31, A_p drawn from 1..8, all 7 metrics, every problem
                     correlated; valid / summary / flags copied to the host;
  fleet-mixed        the same with every second problem correlated (the others diagonal);
  fleet-corr-detail  P = 256 x 300 x 31, every problem correlated, pair + step copied to the host as well.
Four paths, alternating in one process, each from float64 host rows in the planner's world frame to host copies of the
results, host clock ending in a synchronise:
  host_call         fo_metric_batch_host_corr: the bundles of all problems in one contiguous float64 array (filled
                    before the clock starts), the agents shifted and concatenated into float32 arrays inside the clock,
                    outputs into arrays allocated once.  Timed with pageable and with page-locked ego rows;
  python_batch      MetricEngine.set_agent_batch(..., vehicles, correlated=True) + assess_batch(per-problem float64
                    arrays) + .cpu() of every output;
  c_loop            a route-B embedder without batches: per problem, fo_metric_batch_host_corr with n_problems = 1 (its
                    float64 rows, its agents to float32) into slices of arrays allocated once.
Outputs are compared bit for bit: host_call against python_batch and the page-locked call, and against c_loop run under
FO_TEAM_WARPS set to the batch's team size (a single problem's results depend on it).

    python scripts/bench_batch_host_corr.py [--steps 10] [--warmup 2] [--workloads fleet-corr,fleet-mixed,fleet-corr-detail]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_batch import gpu_info, problems, team_warps  # noqa: E402
from bench_batch_corr import correlate  # noqa: E402
from bench_batch_host import agents_f32, far, params_of  # noqa: E402
from bench_batch_vehicles import fleet  # noqa: E402


def cov_f32(ags):
    """cov_xy rows of the given problems, concatenated as agents_f32 concatenates their agents (zero where diagonal)."""
    A, S = sum(a.n_agents for a in ags), max([a.t_stride for a in ags], default=0)
    cov = np.zeros((A, S), np.float32)
    a0 = 0
    for ag in ags:
        if ag.cov_xy is not None:
            cov[a0:a0 + ag.n_agents, :ag.t_stride] = ag.cov_xy
        a0 += ag.n_agents
    return cov


def bench(name, probs, case, vehicles, detail, steps, warmup, sms):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import MetricEngine, vehicle_struct
    sync = torch.cuda.synchronize
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    ags, orgs, egos = [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs]
    P, T = len(probs), int(egos[0].shape[1])
    counts = np.array([len(e) for e in egos], np.int64)
    offs = np.concatenate([[0], np.cumsum(counts)])
    N = int(offs[-1])
    n_ag = np.array([a.n_agents for a in ags], np.int64)
    pairs = int(np.dot(counts, n_ag))
    pair_offs = np.concatenate([[0], np.cumsum(counts * n_ag)])
    ego64 = np.concatenate(egos)                                   # the planner's output buffer
    ego64_pinned = torch.from_numpy(ego64).pin_memory().numpy()
    org = np.asarray(orgs, np.float64)
    veh = (L.FoVehicle * P)(*[vehicle_struct(v) for v in vehicles])
    corr = np.array([a.cov_xy is not None for a in ags], np.uint8)
    prm = params_of(eng, L)
    problems_c = (L.FoBatchProblem * P)()
    for p in range(P):
        problems_c[p].traj_begin, problems_c[p].n_traj = int(offs[p]), int(counts[p])
        problems_c[p].n_agents, problems_c[p].t_stride = ags[p].n_agents, ags[p].t_stride
    fields = ("valid", "flags", "summary") + (("pair", "step") if detail else ())

    def outputs():
        o = {"valid": np.empty(N, np.uint8), "flags": np.empty(N, np.uint32), "summary": np.empty((N, 10), np.float32)}
        if detail:
            o["pair"] = np.empty(pairs * L.FO_PAIR_K, np.float32)
            o["step"] = np.empty(pairs * (T - 1) * L.FO_STEP_K, np.float32)
        return o
    out_h, out_l = outputs(), outputs()
    ptr = lambda o, k, off=0: o[k][off:].ctypes.data if k in o else None  # noqa: E731

    def host_call(ego):
        raw, keep = agents_f32(L, ags, orgs)
        cov = cov_f32(ags)
        L.check(L.lib.fo_metric_batch_host_corr(ego.ctypes.data, N, T, org.ctypes.data, C.byref(raw), cov.ctypes.data,
                                                P, problems_c, corr.ctypes.data, veh, C.byref(prm), ptr(out_h, "valid"),
                                                ptr(out_h, "summary"), ptr(out_h, "flags"), ptr(out_h, "pair"),
                                                ptr(out_h, "step")), "fo_metric_batch_host_corr")
        return out_h

    def python_batch():
        eng.set_agent_batch(ags, orgs, vehicles=vehicles, correlated=True)
        r = eng.assess_batch(egos, want_pair=detail, want_step=detail)
        o = {"valid": r.valid.cpu().numpy(), "flags": r.flags.cpu().numpy().view(np.uint32),
             "summary": r.summary.cpu().numpy()}
        if detail:
            o["pair"], o["step"] = r.pair.cpu().numpy(), r.step.cpu().numpy()
        return o

    one = (L.FoBatchProblem * 1)()

    def c_loop():
        for p in range(P):
            lo, n = int(offs[p]), int(counts[p])
            raw, keep = agents_f32(L, ags[p:p + 1], orgs[p:p + 1])
            cov = cov_f32(ags[p:p + 1])
            one[0].traj_begin, one[0].n_traj, one[0].n_agents, one[0].t_stride = 0, n, ags[p].n_agents, ags[p].t_stride
            q = int(pair_offs[p])
            L.check(L.lib.fo_metric_batch_host_corr(ego64[lo:].ctypes.data, n, T, org[p:].ctypes.data, C.byref(raw),
                                                    cov.ctypes.data, 1, one, corr[p:].ctypes.data, C.byref(veh[p]),
                                                    C.byref(prm), ptr(out_l, "valid", lo), ptr(out_l, "summary", lo),
                                                    ptr(out_l, "flags", lo), ptr(out_l, "pair", q * L.FO_PAIR_K),
                                                    ptr(out_l, "step", q * (T - 1) * L.FO_STEP_K)),
                    "fo_metric_batch_host_corr")
        return out_l

    paths = {"host_call": lambda: host_call(ego64), "host_call_pinned": lambda: host_call(ego64_pinned),
             "python_batch": python_batch, "c_loop": c_loop}
    times = {k: [] for k in paths}
    for k, fn in paths.items():
        for _ in range(warmup):
            fn()
    sync()
    for _ in range(2):                         # alternate the paths, twice
        for k, fn in paths.items():
            for _ in range(steps):
                t0 = time.perf_counter()
                fn()
                sync()
                times[k].append((time.perf_counter() - t0) * 1e3)

    got = {k: v.copy() for k, v in host_call(ego64).items()}
    same = lambda a, b: all(np.array_equal(a[f], b[f], equal_nan=True) and a[f].shape == b[f].shape  # noqa: E731
                            for f in fields)
    eq_py = same(got, python_batch())
    got_pinned = {k: v.copy() for k, v in host_call(ego64_pinned).items()}
    W = team_warps(N, T, int(n_ag.min()), sms)
    os.environ["FO_TEAM_WARPS"] = str(W)
    eq_loop = same(got, c_loop())
    del os.environ["FO_TEAM_WARPS"]
    med = lambda x: float(np.median(x))  # noqa: E731
    rng = lambda x: [min(x), max(x)]  # noqa: E731
    res = {"workload": name, "P": P, "N_total": N, "T": T, "detail": detail, "pairs": pairs,
           "correlated_problems": int(corr.sum()), "ego_f64_MB": N * T * 5 * 8 / 1e6, "team_warps": W,
           "outputs_equal_python_batch": bool(eq_py), "outputs_equal_c_loop": bool(eq_loop),
           "outputs_equal_pinned": bool(same(got, got_pinned))}
    for k, v in times.items():
        res[k + "_ms"], res[k + "_ms_range"] = med(v), rng(v)
    res["python_batch_over_host_call_pinned"] = med(times["python_batch"]) / med(times["host_call_pinned"])
    res["c_loop_over_host_call_pinned"] = med(times["c_loop"]) / med(times["host_call_pinned"])
    return res


def card():
    """gpu_info(), with the power limit read through nvidia-smi's query interface when NVML is not importable."""
    info = gpu_info()
    if info.get("power_limit_w") is None:
        try:
            q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip().split(",")
            info["power_limit_w"], info["power_limit_source"] = float(q[1]), "nvidia-smi"
        except Exception as e:                  # reported, not guessed
            info["power_limit_query_error"] = repr(e)
    return info


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
        sys.exit("bench_batch_host_corr.py needs a CUDA device")
    info = card()
    res = {"gpu": info, "results": []}
    for wl in args.workloads.split(","):
        if wl in ("fleet-corr", "fleet-mixed"):
            probs, case = problems(256, 1000, 31, lambda r: r.integers(1, 9), seed=1)
            every, vehicles, detail, seed = (1 if wl == "fleet-corr" else 2), fleet(256, 1), False, 1
        elif wl == "fleet-corr-detail":
            probs, case = problems(256, 300, 31, lambda r: r.integers(1, 9), seed=3)
            every, vehicles, detail, seed = 1, fleet(256, 3), True, 3
        else:
            ap.error(f"unknown workload {wl}")
        rng = np.random.default_rng(11)
        probs = [((correlate(ag, rng) if p % every == 0 else ag), o, e) for p, (ag, o, e) in enumerate(probs)]
        res["results"].append(bench(wl, far(probs, seed), case, vehicles, detail, args.steps, args.warmup, info["sms"]))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
