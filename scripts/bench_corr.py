"""Cost of correlated prediction covariances: fo_metric_bundle_corr against fo_metric_bundle; prints one JSON line.

Both paths assess the same seeded bundle and agents.  The correlated set has var_x != var_y per state (the synthetic
variance times U(0.3, 3) per axis) and rho ~ U(-0.9, 0.9); the diagonal set has the same variances and rho = 0, so the
two differ only in the CP function and its table section.  Workloads:
  c-lat         1 k x 32 agents x 31 states (30 steps), all 7 metrics -- the per-planning-step latency shape;
  sweep         1 M x 256 x 51, all 7 metrics -- the throughput shape (one-warp window filter);
  sweep-detail  10 k x 256 x 51 with pair and step outputs (the detail kernel; 1 M rows of step output would not fit).
Kernel time: CUDA events around each metric call on a device-resident bundle, the two paths alternating, after warm-up;
median and range over the steps.  n_cp is the number of CP evaluations of one pass (fo_metric_stats on the diagonal
path: the 5 m gate does not depend on the covariance), so (t_corr - t_diag) / n_cp is the added time per gated step.

    python scripts/bench_corr.py [--steps 5] [--warmup 2] [--workloads c-lat,sweep,sweep-detail]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {"c-lat": (1000, 32, 31, False), "sweep": (1_000_000, 256, 51, False), "sweep-detail": (10_000, 256, 51, True)}


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


def agent_sets(n_agents, n_states, seed):
    """(correlated, diagonal) AgentSets of the same agents and variances."""
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    rng = np.random.default_rng(seed)
    agents = S.agent_table(n_agents, n_states, rng=rng)
    corr, diag = [], []
    for a in agents:
        v = np.asarray(a["var"])
        vx, vy = v * rng.uniform(0.3, 3.0, n_states), v * rng.uniform(0.3, 3.0, n_states)
        c = rng.uniform(-0.9, 0.9, n_states) * np.sqrt(vx * vy)
        for out, cxy in ((corr, c), (diag, 0.0 * c)):
            b = dict(a)
            b["cov"] = np.stack((np.stack((vx, cxy), -1), np.stack((cxy, vy), -1)), -2)
            out.append(b)
    return AgentSet.from_case(corr), AgentSet.from_case(diag)


def run(name, n_traj, n_agents, n_states, detail, steps, warmup):
    import torch
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import BundleResult, MetricEngine
    dev = torch.device("cuda:0")
    corr, diag = agent_sets(n_agents, n_states, seed=7)
    assert corr.cov_xy is not None and diag.cov_xy is None
    engines = {}
    for key, ag in (("corr", corr), ("diag", diag)):
        e = MetricEngine(S.VEHICLE, 0.1, S.ALL_METRICS, S.DEFAULT_THRESHOLDS)
        e.set_agents(ag)
        engines[key] = e
    ego = engines["diag"].to_device_bundle(S.ego_bundle(n_traj, n_states, seed=11))
    N, A, T = n_traj, n_agents, n_states
    outs = {}
    for key in engines:
        o = BundleResult(torch.empty(N, dtype=torch.uint8, device=dev), torch.empty((N, 10), dtype=torch.float32, device=dev),
                         torch.empty(N, dtype=torch.int32, device=dev))
        if detail:
            o.pair = torch.empty((N, A, 12), dtype=torch.float32, device=dev)
            o.step = torch.empty((N, A, T - 1, 3), dtype=torch.float32, device=dev)
        outs[key] = o
    times = {"corr": [], "diag": []}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(warmup + steps):
        for key in ("diag", "corr"):
            ev0.record()
            engines[key].assess(ego, out=outs[key])
            ev1.record()
            torch.cuda.synchronize()
            if it >= warmup:
                times[key].append(ev0.elapsed_time(ev1))
    res = {"workload": name, "shape": [N, A, T], "detail": detail}
    for key, t in times.items():
        res[key + "_ms"] = {"median": float(np.median(t)), "min": float(min(t)), "max": float(max(t))}
    n_cp = engines["diag"].work_stats(ego[:min(N, 100_000)])["cp"] * (N / min(N, 100_000))
    res["n_cp"] = float(n_cp)
    dt = res["corr_ms"]["median"] - res["diag_ms"]["median"]
    res["added_ns_per_cp"] = dt * 1e6 / n_cp if n_cp else None
    res["valid_equal"] = bool(torch.equal(outs["corr"].valid, outs["diag"].valid))
    res["cp_max_corr_diag"] = [float(outs["corr"].summary[:, 4].max()), float(outs["diag"].summary[:, 4].max())]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_corr.py needs a CUDA device")
    out = {"gpu": gpu_info(), "results": []}
    for name in args.workloads.split(","):
        out["results"].append(run(name, *WORKLOADS[name], steps=args.steps, warmup=args.warmup))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
