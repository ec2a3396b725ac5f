"""Correlated prediction covariances in trajectory-sharded sweeps and in the work counters: fo_metric_bundle_corr_peers
(the fused result exchange of parallel.PeerResultGatherer on a correlated table), fo_metric_stats_corr and
MetricEngine.work_stats(correlated=True).

CPU: declarations and exports, argument checks that need no device, code-size budgets of the new kernels.  GPU (-m gpu):
two ranks sharing one GPU exchange a correlated bundle through peer-mapped buffers and through the plain all-gather, and
assemble what fo_metric_bundle_corr gives for the whole bundle, bit for bit; fo_metric_bundle_corr_peers without peers
is fo_metric_bundle_corr; the counters of a correlated table equal those of the diagonal table of the same agents, and
the counter pass writes the outputs of fo_metric_bundle_corr."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import corr_oracle as CO
from kernel_sizes import size_of
from frenetix_occlusion_b200 import synthetic as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARMED = {"harm": 0.1, "risk": 0.01, "be": 1.0, "cp": 0.05, "ttc": 2.0, "wttc": None, "ttce": None, "dce": 2.0}
FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_new_calls_are_declared_and_exported():
    from frenetix_occlusion_b200 import _lib as L
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fo_b200.h")).read(), flags=re.S)
    for name in ("fo_metric_bundle_corr_peers", "fo_metric_stats_corr"):
        assert re.search(r"\b%s\s*\(" % name, text), name
        assert name in L.EXPORTED_SYMBOLS and hasattr(L.lib, name)


def _args(**kw):
    from frenetix_occlusion_b200 import _lib as L
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    a = L.FoMetricArgs()
    a.n_traj, a.n_states, a.ego, a.valid, a.summary, a.flags = 4, 31, p, p, p, p
    for k, v in kw.items():
        setattr(a, k, p if v is True else v)
    return a, buf


def test_peer_call_checks_its_arguments_without_device():
    """The n_peers checks of fo_metric_bundle_corr_peers run before any device query."""
    from frenetix_occlusion_b200 import _lib as L
    f = L.lib.fo_metric_bundle_corr_peers
    for n in (-1, L.FO_MAX_PEERS + 1):
        a, _ = _args(n_peers=n)
        assert f(C.byref(a), None) == FO_ERR_INVALID_ARG, n
        assert b"fo_metric_bundle_corr_peers: n_peers" in L.lib.fo_last_error()
    for out in ("pair", "step"):
        a, _ = _args(n_peers=1, **{out: True})
        assert f(C.byref(a), None) == FO_ERR_UNSUPPORTED, out
        assert b"summary path only" in L.lib.fo_last_error()
    assert f(None, None) == FO_ERR_INVALID_ARG
    a, _ = _args(n_peers=0, n_traj=-1)                  # n_peers = 0: fo_metric_bundle_corr's checks
    assert f(C.byref(a), None) == FO_ERR_INVALID_ARG
    a, _ = _args(n_peers=1)                             # the refusal of fo_metric_bundle_corr stays
    assert L.lib.fo_metric_bundle_corr(C.byref(a), None) == FO_ERR_UNSUPPORTED


def test_stats_call_checks_its_arguments_without_device():
    from frenetix_occlusion_b200 import _lib as L
    f = L.lib.fo_metric_stats_corr
    a, buf = _args()
    assert f(C.byref(a), None, None) == FO_ERR_INVALID_ARG
    assert b"fo_metric_stats_corr: counters_dev" in L.lib.fo_last_error()
    for out in ("pair", "step"):
        a, buf = _args(**{out: True})
        assert f(C.byref(a), C.cast(buf, C.c_void_p), None) == FO_ERR_INVALID_ARG, out
        assert b"summary outputs only" in L.lib.fo_last_error()


def test_correlated_counter_kernels_stay_inside_their_code_size_budgets():
    """The counter kernels are fo_metric_sweep_corr_kernel plus the increments and the epilogue's atomics.  Budgets: the
    sizes measured when they were added (DESIGN.md 5.13) plus 4 kB."""
    budget = {"ILb1ELb0E": 77.375,      # one-warp window-filter shape
              "ILb1ELb1E": 90.0,        # ... with the float64 tie path
              "ILb0ELb0E": 86.625,      # team shape
              "ILb0ELb1E": 102.375}
    for tmpl, kb in budget.items():
        size = size_of("fo_metric_sweep_corr_stats_kernel", tmpl)
        assert size <= (kb + 4) * 1024, (tmpl, size)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _worker(rank, world, port, peer, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import corr_oracle as CO
        from frenetix_occlusion_b200 import _lib as L
        from frenetix_occlusion_b200 import synthetic as S
        from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
        from frenetix_occlusion_b200.parallel import PeerResultGatherer, ResultGatherer
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        dev = torch.device("cuda", 0)
        torch.cuda.set_device(dev)
        n_total, block = 3000, 256
        g = (PeerResultGatherer if peer else ResultGatherer)(n_total, L.FO_SUMMARY_K, dev, block=block)
        report = []
        for step in range(3):                       # three steps: both buffers of the peer form, and the first one reused
            case = CO.add_correlations(S.make_case(n_total, 24, 31, seed=100 + step), 100 + step)
            eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"], device=dev)
            eng.set_agents(AgentSet.from_case(case["agents"]))
            assert eng._corr
            ego = torch.from_numpy(case["ego"].astype(np.float32)).to(dev)
            ref = eng.assess(ego)                   # fo_metric_bundle_corr on the whole bundle: what the exchange must give
            mine = torch.from_numpy(g.index[rank]).to(dev)
            out = g.local_result()
            assert bool(out.peer_delta) == peer and (not peer or len(out.peer_delta) == world - 1)
            half = len(mine) // 2                   # two launches into slices of the same buffer (bench.py's e2e chunks)
            eng.assess(ego[mine[:half]].contiguous(), out=g.slice_of(out, 0, half))
            eng.assess(ego[mine[half:]].contiguous(), out=g.slice_of(out, half, len(mine)))
            g.gather()
            v, s, f = g.assembled()
            torch.cuda.synchronize()
            report.append((bool(torch.equal(v, ref.valid)), bool(torch.equal(s.view(torch.int32), ref.summary.view(torch.int32))),
                           bool(torch.equal(f, ref.flags)), int(ref.valid.sum())))
        dist.barrier()
        if peer:
            g.close()
        q.put((rank, report, None))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, None, traceback.format_exc() + repr(e)))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("peer", [True, False], ids=["peer", "all_gather"])
def test_sharded_correlated_bundle_assembles_the_whole_bundle(peer, cuda_device):
    import socket
    with socket.socket() as sock:                       # a free rendezvous port
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, peer, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, report, err in res:
        assert err is None, err
        assert all(a and b and c for a, b, c, _ in report), (rank, report)
        assert all(0 < nv < 3000 for *_, nv in report), report      # non-trivial masks


def _engine(case, agents):
    from frenetix_occlusion_b200.engine import MetricEngine
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(agents)
    return eng


def _outputs(eng, t, fn, *extra):
    """valid / summary bits / flags of one direct C call on the engine's table."""
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import BundleResult
    N = int(t.shape[0])
    out = BundleResult(torch.full((N,), 7, dtype=torch.uint8, device=t.device),
                       torch.full((N, L.FO_SUMMARY_K), -3.0, dtype=torch.float32, device=t.device),
                       torch.full((N,), -5, dtype=torch.int32, device=t.device))
    a = eng._args(t, out)
    L.check(getattr(L.lib, fn)(C.byref(a), *extra, eng._stream()), fn)
    torch.cuda.synchronize()
    return out.valid.cpu().numpy(), out.summary.view(torch.int32).cpu().numpy(), out.flags.cpu().numpy()


def _equal(x, y):
    return all(np.array_equal(a, b) for a, b in zip(x, y))


# (seed, N, A, T, metrics, thresholds, FO_TEAM_WARPS): W = 1 with >= 17 agents is the one-warp window-filter shape, the
# rest the team shape; null thresholds run the kernels without the tie path, armed ones with it
SHAPES = [(1, 400, 40, 31, None, None, "1"), (2, 400, 40, 51, None, ARMED, "1"),
          (3, 200, 5, 31, None, None, None), (4, 200, 5, 51, S.DEFAULT_METRICS, ARMED, "2")]


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,a,t,metrics,thr,warps", SHAPES)
def test_peer_call_without_peers_is_the_correlated_call(seed, n, a, t, metrics, thr, warps, cuda_device, monkeypatch):
    from frenetix_occlusion_b200.engine import AgentSet
    if warps:
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
    case = CO.add_correlations(S.make_case(n, a, t, seed=seed, activated_metrics=metrics, thresholds=thr), seed)
    eng = _engine(case, AgentSet.from_case(case["agents"]))
    assert eng._corr
    ego = eng.to_device_bundle(case["ego"])
    ref = _outputs(eng, ego, "fo_metric_bundle_corr")
    got = _outputs(eng, ego, "fo_metric_bundle_corr_peers")
    assert _equal(got, ref)


# A in {1, 40, 300} x T in {2, 31, 51, 128}; the window-filter shape (W = 1, >= 17 agents), the one-warp team shape
# (W = 1, fewer agents) and multi-warp team shapes, BE on (all 7 metrics) and off (the default set), null and armed
# thresholds
COUNTER_CASES = [(11, 300, 1, 31, None, None, "1"), (12, 200, 1, 128, S.DEFAULT_METRICS, ARMED, "1"),
                 (13, 300, 40, 2, None, ARMED, "1"), (14, 300, 40, 51, None, None, "1"),
                 (15, 150, 40, 128, S.DEFAULT_METRICS, None, "8"), (16, 120, 40, 31, None, ARMED, "2"),
                 (17, 80, 300, 51, None, ARMED, "1"), (18, 80, 300, 31, S.DEFAULT_METRICS, None, "1"),
                 (19, 60, 300, 2, None, None, "1"), (20, 60, 300, 128, None, ARMED, "4")]
# With W > 1 the team pools its warps' queue leftovers and lists its BE pairs in shared memory in the order the warps
# arrive (atomicAdd), so which warp drains which item, and with it what each warp's running bounds prune, varies from
# run to run: the box distances, LR4S logits, BE pairs before a range error and BE probes counted there are not
# reproducible even on the diagonal path.  These counters do not depend on that order.
ORDER_FREE = ("visited", "cp", "windows", "windows_kept", "be_nodes", "be_path_chunks")


@pytest.mark.gpu
@pytest.mark.parametrize("nan_cov", [False, True], ids=["pd", "rho1.5"])
@pytest.mark.parametrize("seed,n,a,t,metrics,thr,warps", COUNTER_CASES)
def test_correlated_counters_equal_the_diagonal_ones(seed, n, a, t, metrics, thr, warps, nan_cov, cuda_device,
                                                      monkeypatch):
    """work_stats(correlated=True) of a correlated set equals work_stats() of the same set with cov_xy = None on every
    counter in the one-warp shapes (on the order-free ones with W > 1), also where a covariance is not positive definite
    (NaN CP values); the counter pass writes the outputs of fo_metric_bundle_corr."""
    from frenetix_occlusion_b200.engine import AgentSet
    monkeypatch.setenv("FO_TEAM_WARPS", warps)
    keys = list(ORDER_FREE) if warps != "1" else None
    case = CO.add_correlations(S.make_case(n, a, t, seed=seed, activated_metrics=metrics, thresholds=thr), seed)
    for ag in case["agents"]:                   # pull the agents onto the ego paths: many gated steps and BE pairs
        ag["pos"] = np.asarray(ag["pos"]) * 0.3
    corr = AgentSet.from_case(case["agents"])
    if nan_cov:                                 # every second agent: |rho| = 1.5 in every state
        corr.cov_xy[::2] = 1.5 * np.sqrt(corr.var_x[::2] * corr.var_y[::2])
    diag = AgentSet.from_case(case["agents"])
    diag.cov_xy = None
    ec, ed = _engine(case, corr), _engine(case, diag)
    assert ec._corr and not ed._corr
    ego = ec.to_device_bundle(case["ego"])
    want = ed.work_stats(ego)
    got = ec.work_stats(ego, correlated=True)
    pick = (lambda d: {k: d[k] for k in keys}) if keys else (lambda d: d)    # noqa: E731
    assert pick(got) == pick(want)
    assert want["cp"] > 0 and want["visited"] > 0
    cnt = torch.zeros(10, dtype=torch.int64, device=ego.device)
    outs = _outputs(ec, ego, "fo_metric_stats_corr", C.c_void_p(cnt.data_ptr()))
    assert pick(dict(zip(want, cnt.cpu().tolist()))) == pick(want)
    ref = _outputs(ec, ego, "fo_metric_bundle_corr")
    assert _equal(outs, ref)
    if nan_cov:
        assert np.isnan(ref[1].view(np.float32)[:, 4]).any()


@pytest.mark.gpu
def test_correlated_flag_without_effect_on_a_diagonal_set(cuda_device, monkeypatch):
    from frenetix_occlusion_b200.engine import AgentSet
    monkeypatch.setenv("FO_TEAM_WARPS", "1")           # a shape whose counters are reproducible (ORDER_FREE)
    case = S.make_case(500, 40, 51, seed=31)
    eng = _engine(case, AgentSet.from_case(case["agents"]))
    assert not eng._corr
    assert eng.work_stats(case["ego"], correlated=True) == eng.work_stats(case["ego"])


@pytest.mark.gpu
def test_correlated_set_without_the_flag_still_raises(cuda_device):
    from frenetix_occlusion_b200.engine import AgentSet
    case = CO.add_correlations(S.make_case(10, 4, 31, seed=29), 29)
    eng = _engine(case, AgentSet.from_case(case["agents"]))
    with pytest.raises(ValueError, match="diagonal"):
        eng.work_stats(case["ego"])
