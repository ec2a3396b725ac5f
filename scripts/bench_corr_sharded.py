"""The correlated C-sweep sharded over N GPUs; rank 0 prints one JSON line.

    torchrun --nproc-per-node N scripts/bench_corr_sharded.py [--steps 5] [--warmup 2] [--exchanges peer,nccl]

Workload: the sweep of scripts/bench_corr.py with correlated covariances, 1 M x 256 x 51, all 7 metrics, rho ~ U(-0.9,
0.9) and var_x != var_y per state (the same seeds).  With N > 1 the bundle is sharded as ``bench.py --gpus N`` shards it:
interleaved blocks of 1024 trajectories, one rank per GPU, the agent table packed on every rank.  Exchanges:
  peer   PeerResultGatherer: the summary kernel's epilogue stores every result row into all ranks' peer-mapped buffers
         (fo_metric_bundle_corr_peers), then a 4-byte all-reduce handshake;
  nccl   ResultGatherer: the kernel writes this rank's slice (fo_metric_bundle_corr), then one all_gather_into_tensor.

Per step: every rank starts behind a barrier, and the step time is the host clock around the metric call, the exchange
and a device synchronise, maximum over ranks.  Kernel time: CUDA events around the metric call on every rank; the spread
is max / mean over the ranks, per step.  The correlated cost gathers at the few per cent of evaluations that reach the CP
drain, so 1024-trajectory blocks may balance worse than they do on diagonal bundles.

Rank 0 first runs the whole bundle through fo_metric_bundle_corr on its own GPU while the other ranks wait: that is the
one-GPU step time of this run (scaling efficiency = t_1 / (N t_N)) and the reference the assembled outputs of every
exchange must equal byte for byte.  It also counts the CP evaluations with work_stats(correlated=True) next to the
diagonal-engine estimate scripts/bench_corr.py uses (a 100 k-trajectory sample scaled to the bundle); the two are equal
because the counters do not depend on the covariances.
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

SHARD_BLOCK = 1024                  # bench.py's interleaved shard block


def gpu_info(index):
    import torch
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["max_sm_clock_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:                      # reported, not guessed
        info["power_limit_w"] = None
        info["power_limit_error"] = repr(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ref-steps", type=int, default=2, help="timed one-GPU steps of the whole bundle on rank 0")
    ap.add_argument("--exchanges", default="peer,nccl")
    ap.add_argument("--n-traj", type=int, default=1_000_000)
    ap.add_argument("--n-agents", type=int, default=256)
    ap.add_argument("--n-states", type=int, default=51)
    ap.add_argument("--stats-sample", type=int, default=100_000)
    ap.add_argument("--backend", default="nccl", choices=["nccl", "gloo"],
                    help="gloo: ranks may share a GPU (a rehearsal of the sharded path; its times are no scaling measurement)")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    import bench_corr
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import BundleResult, MetricEngine
    from frenetix_occlusion_b200.parallel import PeerResultGatherer, ResultGatherer, shard_indices

    if not torch.cuda.is_available():
        raise SystemExit("bench_corr_sharded.py needs CUDA devices")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.backend == "gloo":
        local %= torch.cuda.device_count()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.backend == "nccl":
            dist.init_process_group("nccl", device_id=dev)
        else:
            dist.init_process_group("gloo")
    N, A, T = args.n_traj, args.n_agents, args.n_states
    evals = N * A * (T - 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    corr, diag = bench_corr.agent_sets(A, T, seed=7)
    assert corr.cov_xy is not None
    eng = MetricEngine(S.VEHICLE, 0.1, S.ALL_METRICS, S.DEFAULT_THRESHOLDS, device=dev)
    eng.set_agents(corr)
    ego_all = S.ego_bundle(N, T, seed=11).astype(np.float32)
    mine = shard_indices(N, world, rank, SHARD_BLOCK) if world > 1 else np.arange(N)
    ego_dev = torch.from_numpy(np.ascontiguousarray(ego_all[mine])).to(dev)

    def new_result(n):
        return BundleResult(torch.empty(n, dtype=torch.uint8, device=dev),
                            torch.empty((n, L.FO_SUMMARY_K), dtype=torch.float32, device=dev),
                            torch.empty(n, dtype=torch.int32, device=dev))

    report = {"workload": "corr-sweep", "shape": [N, A, T], "evaluations": evals, "gpus": world, "backend": args.backend,
              "gpu": [None] * world, "steps": args.steps, "warmup": args.warmup}
    info = gpu_info(local)
    if world > 1:
        dist.all_gather_object(report["gpu"], info)
    else:
        report["gpu"] = [info]

    # ---- rank 0: the whole bundle on one GPU (fo_metric_bundle_corr), the reference outputs and the counters --------
    ref_bytes = None
    if rank == 0:
        full = torch.from_numpy(ego_all).to(dev)
        ref = new_result(N)
        host_ms, kern_ms = [], []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(1 + args.ref_steps):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            e0.record()
            eng.assess(full, out=ref)
            e1.record()
            torch.cuda.synchronize(dev)
            if i > 0:
                host_ms.append((time.perf_counter() - t0) * 1e3)
                kern_ms.append(e0.elapsed_time(e1))
        ref_bytes = (ref.valid.cpu().numpy().tobytes(), ref.summary.view(torch.int32).cpu().numpy().tobytes(),
                     ref.flags.cpu().numpy().tobytes())
        t1 = float(np.median(host_ms))
        report["one_gpu"] = {"step_ms": t1, "step_ms_range": [min(host_ms), max(host_ms)],
                             "kernel_ms": float(np.median(kern_ms)), "evals_per_s": evals / (t1 * 1e-3),
                             "valid": int(ref.valid.sum())}
        # CP evaluations: work_stats(correlated=True) and the diagonal-engine estimate of bench_corr.py, on the same
        # sample; then both on the whole bundle
        ed = MetricEngine(S.VEHICLE, 0.1, S.ALL_METRICS, S.DEFAULT_THRESHOLDS, device=dev)
        ed.set_agents(diag)
        m = min(N, args.stats_sample)
        sample_corr = eng.work_stats(full[:m], correlated=True)
        sample_diag = ed.work_stats(full[:m])
        whole_corr = eng.work_stats(full, correlated=True)
        whole_diag = ed.work_stats(full)
        report["n_cp"] = {"sample": m,
                          "corr_work_stats_scaled": sample_corr["cp"] * (N / m),
                          "diag_estimate_bench_corr": sample_diag["cp"] * (N / m),
                          "corr_work_stats_whole": whole_corr["cp"], "diag_work_stats_whole": whole_diag["cp"],
                          "all_counters_equal": sample_corr == sample_diag and whole_corr == whole_diag}
        del full, ref
        torch.cuda.empty_cache()
    barrier()

    # ---- the sharded sweep, per exchange ---------------------------------------------------------------------------
    report["runs"] = []
    for exchange in (args.exchanges.split(",") if world > 1 else []):
        g = (PeerResultGatherer if exchange == "peer" else ResultGatherer)(N, L.FO_SUMMARY_K, dev, block=SHARD_BLOCK)
        assert g.counts[rank] == len(mine)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def step():
            out = g.local_result()
            e0.record()
            eng.assess(ego_dev, out=out)
            e1.record()
            g.gather()

        for _ in range(args.warmup):
            step()
        times = []
        for _ in range(args.steps):
            barrier()
            t0 = time.perf_counter()
            step()
            torch.cuda.synchronize(dev)
            times.append(((time.perf_counter() - t0) * 1e3, e0.elapsed_time(e1)))
        mine_t = torch.tensor(times, dtype=torch.float64, device=dev)               # [steps, 2]
        every = torch.empty(world * mine_t.numel(), dtype=torch.float64, device=dev)  # flat: gloo takes no stacked form
        dist.all_gather_into_tensor(every, mine_t.flatten())
        every = every.view(world, *mine_t.shape).cpu().numpy()                       # [world, steps, 2]
        step_ms = every[:, :, 0].max(axis=0)                                          # slowest rank, per step
        kern = every[:, :, 1]
        spread = kern.max(axis=0) / kern.mean(axis=0)
        run = {"exchange": exchange, "step_ms": float(np.median(step_ms)),
               "step_ms_range": [float(step_ms.min()), float(step_ms.max())],
               "evals_per_s": evals / (float(np.median(step_ms)) * 1e-3),
               "kernel_ms_per_rank": [float(np.median(kern[r])) for r in range(world)],
               "kernel_spread_max_over_mean": float(np.median(spread)),
               "kernel_spread_range": [float(spread.min()), float(spread.max())]}
        if rank == 0:
            v, s, f = g.assembled()
            got = (v.cpu().numpy().tobytes(), s.view(torch.int32).cpu().numpy().tobytes(), f.cpu().numpy().tobytes())
            run["outputs_identical_to_one_gpu"] = got == ref_bytes
            run["scaling_efficiency"] = report["one_gpu"]["step_ms"] / (world * run["step_ms"])
        report["runs"].append(run)
        barrier()
        if exchange == "peer":
            g.close()
        del g
    if rank == 0:
        print(json.dumps(report), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
