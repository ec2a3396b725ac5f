"""A batch of planning problems from host memory in one C-ABI call (fo_metric_batch_host) against the two ways a host
caller had before; prints one JSON line.

Workloads (seeded, the problems and mixed fleet of scripts/bench_batch_vehicles.py, every problem moved by its own
UTM-sized offset of 1e5-6e6 m so the float64 origin shift is real work):
  fleet         P = 256 problems x 1000 trajectories x T = 31, A_p drawn from 1..8, all 7 metrics, one vehicle per
                problem; valid / summary / flags copied to the host;
  fleet-detail  P = 256 x 300 x 31, the same with pair + step copied to the host as well.
Three paths, alternating in one process, each from float64 host arrays in the planner's world frame to host copies of
the results, host clock ending in a synchronise:
  host_call     fo_metric_batch_host: the bundles of all problems in one contiguous float64 array (the planner's output
                buffer, filled before the clock starts; concat_ms is what np.concatenate of per-problem arrays would
                add), the agents shifted and concatenated into float32 arrays inside the clock, outputs into arrays
                allocated once.  Timed with pageable and with page-locked ego rows;
  python_batch  MetricEngine.set_agent_batch(..., vehicles) + assess_batch(per-problem float64 arrays) + .cpu() of
                every output;
  c_loop        what a ctypes embedder without torch runs today: per problem, numpy shift of its bundle to float32,
                its agents to float32, fo_metric_bundle_host with its vehicle, into slices of arrays allocated once.
Outputs are compared bit for bit: host_call against python_batch, and against c_loop run under FO_TEAM_WARPS set to the
batch's team size (the summary results of fo_metric_bundle depend on it).  A separate torch.profiler pass over two
host calls gives the time of fo_ego_ingest_kernel and of the host-to-device copies, and their rates.

    python scripts/bench_batch_host.py [--steps 10] [--warmup 2] [--workloads fleet,fleet-detail]
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

from bench_batch import gpu_info, problems, team_warps  # noqa: E402
from bench_batch_vehicles import fleet  # noqa: E402


def far(probs, seed):
    rng = np.random.default_rng(seed)
    out = []
    for ag, origin, ego in probs:
        dx, dy = rng.uniform(1e5, 6e6, 2)
        ego = ego.astype(np.float64)
        ego[..., 0] += dx
        ego[..., 1] += dy
        live = np.arange(ag.t_stride)[None, :] < ag.n_states[:, None]
        ag.x, ag.y = ag.x + dx * live, ag.y + dy * live
        out.append((ag, (origin[0] + dx, origin[1] + dy), ego))
    return out


def params_of(eng, L):
    a = L.FoMetricArgs()
    a.vehicle, a.harm, a.dt = eng.vehicle, eng.harm, eng.dt
    a.metric_mask, a.threshold_mask = eng.metric_mask, eng.threshold_mask
    for name in L.T_BITS:
        v = eng.thresholds.get(name)
        setattr(a, "thr_" + name, float(v) if v is not None else 0.0)
    return a


def agents_f32(L, ags, orgs):
    """FoAgentsRaw with HOST pointers: the agents of the given problems concatenated, shifted in float64, float32."""
    A, S = sum(a.n_agents for a in ags), max([a.t_stride for a in ags], default=0)
    fl = np.zeros((6, A, S), np.float32)
    pa = np.empty((4, A), np.float32)
    ia = np.empty((2, A), np.int32)
    a0 = 0
    for ag, o in zip(ags, orgs):
        n, tp = ag.n_agents, ag.t_stride
        r = slice(a0, a0 + n)
        fl[0, r, :tp], fl[1, r, :tp] = ag.x - o[0], ag.y - o[1]
        fl[2, r, :tp], fl[3, r, :tp], fl[4, r, :tp], fl[5, r, :tp] = ag.yaw, ag.v, ag.var_x, ag.var_y
        pa[:, r] = (ag.length, ag.width, ag.buf_length, ag.buf_width)
        ia[:, r] = (ag.n_states, ag.kind)
        a0 += n
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = A, S
    raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y = [fl[i].ctypes.data for i in range(6)]
    raw.length, raw.width, raw.buf_length, raw.buf_width = [pa[i].ctypes.data for i in range(4)]
    raw.n_states, raw.kind = ia[0].ctypes.data, ia[1].ctypes.data
    return raw, (fl, pa, ia)


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
    t0 = time.perf_counter()
    ego64 = np.concatenate(egos)                                   # the planner's output buffer
    concat_ms = (time.perf_counter() - t0) * 1e3
    ego64_pinned = torch.from_numpy(ego64).pin_memory().numpy()
    org = np.asarray(orgs, np.float64)
    veh = (L.FoVehicle * P)(*[vehicle_struct(v) for v in vehicles])
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
        L.check(L.lib.fo_metric_batch_host(ego.ctypes.data, N, T, org.ctypes.data, C.byref(raw), P, problems_c, veh,
                                           C.byref(prm), ptr(out_h, "valid"), ptr(out_h, "summary"),
                                           ptr(out_h, "flags"), ptr(out_h, "pair"), ptr(out_h, "step")),
                "fo_metric_batch_host")
        return out_h

    def python_batch():
        eng.set_agent_batch(ags, orgs, vehicles=vehicles)
        r = eng.assess_batch(egos, want_pair=detail, want_step=detail)
        o = {"valid": r.valid.cpu().numpy(), "flags": r.flags.cpu().numpy().view(np.uint32),
             "summary": r.summary.cpu().numpy()}
        if detail:
            o["pair"], o["step"] = r.pair.cpu().numpy(), r.step.cpu().numpy()
        return o

    def c_loop():
        for p in range(P):
            lo, n = int(offs[p]), int(counts[p])
            e32 = (egos[p] - np.array([orgs[p][0], orgs[p][1], 0, 0, 0])).astype(np.float32)
            raw, keep = agents_f32(L, ags[p:p + 1], orgs[p:p + 1])
            prm.vehicle = veh[p]
            q = int(pair_offs[p])
            L.check(L.lib.fo_metric_bundle_host(e32.ctypes.data, n, T, C.byref(raw), C.byref(prm),
                                                ptr(out_l, "valid", lo), ptr(out_l, "summary", lo),
                                                ptr(out_l, "flags", lo), ptr(out_l, "pair", q * L.FO_PAIR_K),
                                                ptr(out_l, "step", q * (T - 1) * L.FO_STEP_K)),
                    "fo_metric_bundle_host")
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

    # outputs: host call vs the Python batch, and vs the loop under the batch's team size
    got = {k: v.copy() for k, v in host_call(ego64).items()}
    same = lambda a, b: all(np.array_equal(a[f], b[f], equal_nan=True) and a[f].shape == b[f].shape  # noqa: E731
                            for f in fields)
    eq_py = same(got, python_batch())
    got_pinned = {k: v.copy() for k, v in host_call(ego64_pinned).items()}
    W = team_warps(N, T, int(n_ag.min()), sms)
    os.environ["FO_TEAM_WARPS"] = str(W)
    eq_loop = same(got, c_loop())
    del os.environ["FO_TEAM_WARPS"]

    # the ingest kernel and the copies, from a profiler pass of their own
    ingest_us, h2d_us, h2d_bytes = [], [], []
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                host_call(ego64_pinned)
            sync()
        for ev in prof.events():
            if "fo_ego_ingest_kernel" in ev.name:
                ingest_us.append(ev.device_time_total)
            elif "Memcpy HtoD" in ev.name:
                h2d_us.append(ev.device_time_total)
        prof_error = None
    except Exception as e:                      # reported, not guessed
        prof_error = repr(e)
    med = lambda x: float(np.median(x))  # noqa: E731
    rng = lambda x: [min(x), max(x)]  # noqa: E731
    ingest_bytes = N * T * 5 * (8 + 4)           # float64 read + float32 written, per call
    res = {"workload": name, "P": P, "N_total": N, "T": T, "detail": detail, "pairs": pairs,
           "ego_f64_MB": N * T * 5 * 8 / 1e6, "team_warps": W, "concat_ms": concat_ms,
           "outputs_equal_python_batch": bool(eq_py), "outputs_equal_c_loop": bool(eq_loop),
           "outputs_equal_pinned": bool(same(got, got_pinned))}
    for k, v in times.items():
        res[k + "_ms"], res[k + "_ms_range"] = med(v), rng(v)
    res["python_batch_over_host_call"] = med(times["python_batch"]) / med(times["host_call"])
    res["c_loop_over_host_call"] = med(times["c_loop"]) / med(times["host_call"])
    if ingest_us:
        per_call = sum(ingest_us) / 2
        res["ingest_kernel_us_per_call"] = per_call
        res["ingest_launches_per_call"] = len(ingest_us) / 2
        res["ingest_GB_per_s"] = ingest_bytes / (per_call * 1e-6) / 1e9
    else:
        res["ingest_kernel_us_per_call"] = None
        res["profiler_error"] = prof_error or "no fo_ego_ingest_kernel in the trace"
    if h2d_us:
        res["h2d_copies_us_per_call_pinned"] = sum(h2d_us) / 2
        res["h2d_ego_GB_per_s_pinned"] = N * T * 5 * 8 / (sum(h2d_us) / 2 * 1e-6) / 1e9
    return res


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
        sys.exit("bench_batch_host.py needs a CUDA device")
    info = gpu_info()
    res = {"gpu": info, "results": []}
    for wl in args.workloads.split(","):
        if wl == "fleet":
            probs, case = problems(256, 1000, 31, lambda r: r.integers(1, 9), seed=1)
            res["results"].append(bench(wl, far(probs, 1), case, fleet(256, 1), False, args.steps, args.warmup,
                                        info["sms"]))
        elif wl == "fleet-detail":
            probs, case = problems(256, 300, 31, lambda r: r.integers(1, 9), seed=3)
            res["results"].append(bench(wl, far(probs, 3), case, fleet(256, 3), True, args.steps, args.warmup,
                                        info["sms"]))
        else:
            ap.error(f"unknown workload {wl}")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
