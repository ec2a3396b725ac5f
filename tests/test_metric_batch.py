"""Batches of independent planning problems (fo_agent_batch_layout, fo_agents_pack_batch, fo_metric_batch,
MetricEngine.set_agent_batch / assess_batch, batch.assess_interfaces).  The CPU part checks the layout, the argument
validation (before any CUDA call) and the code size of the batched kernels; the GPU part checks that every problem of a
batch gets exactly what the single-problem path gives it."""
import ctypes as C
import os
import random

import numpy as np
import pytest

from conftest import GOLDEN
from kernel_sizes import size_of

FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2


# ---------------------------------------------------------------------------------------------------- CPU
def test_batch_layout_is_aligned_and_disjoint():
    from frenetix_occlusion_b200 import _lib as L
    A = np.array([3, 0, 33, 1, 0, 300, 17], dtype=np.int32)
    Tp = np.array([31, 0, 51, 2, 31, 128, 7], dtype=np.int32)
    off = np.zeros(len(A), dtype=np.int64)
    total = L.lib.fo_agent_batch_layout(len(A), A.ctypes.data, Tp.ctypes.data, off.ctypes.data)
    end = 0
    for p in range(len(A)):
        size = L.lib.fo_agent_table_bytes(int(A[p]), int(Tp[p])) if A[p] else 0
        assert off[p] % 16 == 0 and off[p] >= end, (p, off[p], end)
        end = off[p] + size
    assert off[1] == off[2] and off[4] == off[5]       # problems without agents take no bytes
    assert end <= total < end + 16
    assert L.lib.fo_agent_batch_layout(0, None, None, None) == 0
    bad = np.array([-1], dtype=np.int32)
    assert L.lib.fo_agent_batch_layout(1, bad.ctypes.data, Tp.ctypes.data, off.ctypes.data) == 0
    long_ = np.array([129], dtype=np.int32)
    assert L.lib.fo_agent_batch_layout(1, A.ctypes.data, long_.ctypes.data, off.ctypes.data) == 0


def _batch_args(L, problems, n_traj, T=31, arena_bytes=1 << 20):
    buf = (C.c_float * 64)()
    a = L.FoMetricBatchArgs()
    a.common.ego = a.common.valid = a.common.agent_table = C.cast(buf, C.c_void_p)
    a.common.n_traj, a.common.n_states = n_traj, T
    arr = (L.FoBatchProblem * max(len(problems), 1))()
    for i, (b, n, na, tp, off) in enumerate(problems):
        arr[i].traj_begin, arr[i].n_traj, arr[i].n_agents, arr[i].t_stride, arr[i].table_offset = b, n, na, tp, off
    a.n_problems, a.problems, a.arena_bytes = len(problems), arr, arena_bytes
    a._keep = (buf, arr)
    return a


def test_batch_argument_validation_without_device():
    from frenetix_occlusion_b200 import _lib as L
    run = lambda a: L.lib.fo_metric_batch(C.byref(a), None)  # noqa: E731
    assert L.lib.fo_metric_batch(None, None) == FO_ERR_INVALID_ARG
    a = _batch_args(L, [], 0)
    a.n_problems = -1
    assert run(a) == FO_ERR_INVALID_ARG
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    a.problems = None
    assert run(a) == FO_ERR_INVALID_ARG
    assert run(_batch_args(L, [(0, 4, 2, 31, 0), (5, 3, 2, 31, 4096)], 8)) == FO_ERR_INVALID_ARG   # gap between rows
    assert run(_batch_args(L, [(4, 3, 2, 31, 0), (0, 4, 2, 31, 4096)], 7)) == FO_ERR_INVALID_ARG   # not in row order
    assert run(_batch_args(L, [(0, 4, 2, 31, 0), (4, 5, 2, 31, 4096)], 8)) == FO_ERR_INVALID_ARG   # rows past n_traj
    assert run(_batch_args(L, [(0, 4, 2, 31, 0)], 6)) == FO_ERR_INVALID_ARG                         # rows left uncovered
    assert run(_batch_args(L, [(0, 4, 2, 31, (1 << 20) - 64)], 4)) == FO_ERR_INVALID_ARG           # table past the arena
    assert run(_batch_args(L, [(0, 4, 2, 31, 8)], 4)) == FO_ERR_INVALID_ARG                         # misaligned table
    assert run(_batch_args(L, [(0, 4, 2, 0, 0)], 4)) == FO_ERR_INVALID_ARG                          # agents, no states
    assert run(_batch_args(L, [(0, 4, 2, 129, 0)], 4)) == FO_ERR_UNSUPPORTED                        # t_stride > FO_MAX_STATES
    assert run(_batch_args(L, [(0, 4, 2, 31, 0)], 4, T=129)) == FO_ERR_UNSUPPORTED                  # T > FO_MAX_STATES
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    a.common.pair = a.common.ego
    assert run(a) == FO_ERR_UNSUPPORTED                                                              # detail outputs
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    a.common.step = a.common.ego
    assert run(a) == FO_ERR_UNSUPPORTED
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    a.common.n_peers = 1
    assert run(a) == FO_ERR_UNSUPPORTED                                                              # peer stores
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    a.common.valid = None
    assert run(a) == FO_ERR_INVALID_ARG
    assert b"fo_metric_batch" in L.lib.fo_last_error()
    assert run(_batch_args(L, [(0, 0, 0, 0, 0)], 0)) == 0                                            # nothing to do
    # the pack call: agent counts must add up, tables must lie in the arena
    raw, veh = L.FoAgentsRaw(), L.FoVehicle()
    raw.n_agents, raw.t_stride = 3, 31
    pr = (L.FoBatchProblem * 2)()
    pr[0].n_agents, pr[0].t_stride, pr[1].n_agents, pr[1].t_stride, pr[1].table_offset = 2, 31, 2, 31, 8192
    arena = C.c_void_p(1 << 20)
    assert L.lib.fo_agents_pack_batch(C.byref(raw), 2, pr, C.byref(veh), arena, 1 << 16, None) == FO_ERR_INVALID_ARG
    raw.n_agents = 4
    assert L.lib.fo_agents_pack_batch(C.byref(raw), 2, pr, C.byref(veh), arena, 8192, None) == FO_ERR_INVALID_ARG
    assert L.lib.fo_agents_pack_batch(C.byref(raw), 2, pr, C.byref(veh), arena, 1 << 16, None) == FO_ERR_INVALID_ARG  # NULL arrays
    assert L.lib.fo_agents_pack_batch(None, 2, pr, C.byref(veh), arena, 1 << 16, None) == FO_ERR_INVALID_ARG


def test_batched_kernels_stay_inside_the_instruction_cache_budget():
    """The batched kernels share the summary kernel's body (DESIGN.md 5.1 and 5.4): they are held to the budgets of
    their single-problem counterparts in test_capi.py."""
    assert size_of("fo_metric_batch_kernel", "ILj127ELb1ELb0E", hot=True) <= 44 * 1024   # all 7 metrics, one-warp window-filter shape
    assert size_of("fo_metric_batch_kernel", "ILj127ELb1ELb1E", hot=True) <= 52 * 1024   # ... with the float64 tie path
    assert size_of("fo_metric_batch_kernel", "ILj111ELb1ELb0E", hot=True) <= 34 * 1024   # default metrics
    assert size_of("fo_metric_batch_kernel", "ILj127ELb0ELb0E", hot=True) <= 56 * 1024   # team shape


# ---------------------------------------------------------------------------------------------------- GPU
A_SET = [0, 1, 2, 3, 5, 8, 16, 17, 32, 33, 64, 300]
N_SET = [0, 1, 5, 64, 500]


def _problems(seed, T, n_problems=None, a_set=A_SET, n_set=N_SET, metrics=None, thresholds=None, varied=False):
    """Seeded problems of synthetic.make_case, each moved to its own place kilometres from the others.  ``varied``:
    synthetic.make_varied_case's turned trajectories and agents of every kind that turn, change speed and carry
    per-axis variances."""
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    rng = np.random.default_rng(seed)
    out = []
    for p in range(n_problems or len(a_set)):
        A = a_set[p % len(a_set)]
        N = n_set[(p * 3 + seed) % len(n_set)]
        case = (S.make_varied_case if varied else S.make_case)(max(N, 1), A, T, seed=seed * 1000 + p,
                                                               activated_metrics=metrics, thresholds=thresholds)
        dx, dy = rng.uniform(-5000.0, 5000.0, 2).round(1)
        ego = case["ego"][:N].copy()
        ego[..., 0] += dx
        ego[..., 1] += dy
        ag = AgentSet.from_case(case["agents"])
        ag.x = ag.x + dx * (np.arange(ag.t_stride)[None, :] < ag.n_states[:, None])
        ag.y = ag.y + dy * (np.arange(ag.t_stride)[None, :] < ag.n_states[:, None])
        origin = (float(ag.x[0, 0]), float(ag.y[0, 0])) if ag.n_agents else (0.0, 0.0)
        out.append((ag, origin, ego, case))
    return out


def _engine(case):
    from frenetix_occlusion_b200.engine import MetricEngine
    return MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])


def _assert_batch_equals_single(problems, monkeypatch, warps):
    import torch
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    eng = _engine(problems[0][3])
    eng.set_agent_batch([p[0] for p in problems], [p[1] for p in problems])
    parts = eng.assess_batch([p[2] for p in problems]).split()
    single = _engine(problems[0][3])
    for i, ((ag, origin, ego, _), got) in enumerate(zip(problems, parts)):
        single.set_agents(ag, origin=origin)
        want = single.assess(ego) if len(ego) else None
        torch.cuda.synchronize()
        if want is None:
            assert got.valid.numel() == 0
            continue
        for f in ("valid", "flags", "summary"):
            g, w = getattr(got, f).cpu().numpy(), getattr(want, f).cpu().numpy()
            assert g.shape == w.shape and np.array_equal(g, w, equal_nan=f == "summary"), (i, f, ag.n_agents, len(ego))
            if f == "summary":
                assert np.array_equal(np.isnan(g), np.isnan(w))


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("warps", [1, 4])
def test_batch_equals_single_problem_path(T, warps, cuda_device, monkeypatch):
    _assert_batch_equals_single(_problems(T, T), monkeypatch, warps)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("warps", [1, 4])
def test_batch_equals_single_problem_path_on_varied_agents(T, warps, cuda_device, monkeypatch):
    _assert_batch_equals_single(_problems(T + 1000, T, varied=True), monkeypatch, warps)


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", [None, "default", ["hr", "cp"], ["dce", "ttc", "wttc"]])
@pytest.mark.parametrize("armed", [False, True])
def test_batch_equals_single_problem_path_metrics_and_thresholds(metrics, armed, cuda_device, monkeypatch):
    from frenetix_occlusion_b200 import synthetic as S
    m = S.DEFAULT_METRICS if metrics == "default" else metrics
    thr = dict(S.DEFAULT_THRESHOLDS, dce=0.5, ttc=1.5, be=0.8) if armed else None
    _assert_batch_equals_single(_problems(7 + armed, 31, metrics=m, thresholds=thr), monkeypatch, 1)


@pytest.mark.gpu
def test_small_batch_picks_a_multi_warp_team(cuda_device, monkeypatch):
    """Without FO_TEAM_WARPS a small batch runs one team launch with W > 1; the per-problem path under that W agrees."""
    import torch
    probs = _problems(11, 51, a_set=[9, 40, 12, 16], n_set=[20, 7, 1, 12])
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = sum(len(p[2]) for p in probs)
    a_min = min(p[0].n_agents for p in probs if len(p[2]))
    lg = next(l for l in range(6) if (1 << l) >= a_min or l == 5)
    W = max(1, min(n_sms * 8 * 4 // N, 51 // (4 * (32 >> lg)), 8))
    assert W > 1
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs])
    parts = eng.assess_batch([p[2] for p in probs]).split()
    torch.cuda.synchronize()
    monkeypatch.setenv("FO_TEAM_WARPS", str(W))
    single = _engine(probs[0][3])
    for (ag, origin, ego, _), got in zip(probs, parts):
        single.set_agents(ag, origin=origin)
        want = single.assess(ego)
        for f in ("valid", "flags", "summary"):
            assert np.array_equal(getattr(got, f).cpu().numpy(), getattr(want, f).cpu().numpy(), equal_nan=True), f


@pytest.mark.gpu
def test_batch_of_device_bundles_equals_host_bundles(cuda_device):
    import torch
    probs = _problems(13, 31, a_set=[2, 33], n_set=[40, 9])
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs])
    r_host = eng.assess_batch([p[2] for p in probs])
    r_dev = eng.assess_batch([torch.from_numpy(p[2]).cuda() for p in probs])
    for f in ("valid", "flags", "summary"):          # NaN where a trajectory is flagged FO_F_BE_RANGE
        assert np.array_equal(getattr(r_host, f).cpu().numpy(), getattr(r_dev, f).cpu().numpy(), equal_nan=True), f
    assert list(r_host.offsets) == [0, len(probs[0][2]), len(probs[0][2]) + len(probs[1][2])]


@pytest.mark.gpu
def test_batch_tables_are_byte_identical_to_single_packs(cuda_device):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    probs = _problems(17, 51, a_set=A_SET, n_set=[1])
    probs[3][0].x = probs[3][0].x[:, :40]       # a shorter table stride than the batch's raw row stride
    for k in ("y", "yaw", "v", "var_x", "var_y"):
        setattr(probs[3][0], k, getattr(probs[3][0], k)[:, :40])
    probs[3][0].n_states = np.minimum(probs[3][0].n_states, 40)
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs])
    arena = eng._batch["arena"]
    single = _engine(probs[0][3])
    for p, (ag, origin, _, _) in enumerate(probs):
        single.set_agents(ag, origin=origin)
        if ag.n_agents == 0:
            continue
        off = eng._batch["problems"][p].table_offset
        n = L.lib.fo_agent_table_bytes(ag.n_agents, ag.t_stride)
        torch.cuda.synchronize()
        assert torch.equal(arena[off:off + n], single._table[:n]), p


@pytest.mark.gpu
def test_every_problem_of_a_mixed_batch_matches_the_oracle(cuda_device, monkeypatch):
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    _assert_every_problem_matches_the_oracle(_problems(23, 31, a_set=[0, 3, 17, 40], n_set=[60, 25, 80, 30]))


@pytest.mark.gpu
def test_every_problem_of_a_mixed_batch_matches_the_oracle_on_varied_agents(cuda_device, monkeypatch):
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    _assert_every_problem_matches_the_oracle(_problems(24, 51, a_set=[0, 5, 17, 40], n_set=[60, 25, 80, 30], varied=True))


def _assert_every_problem_matches_the_oracle(probs):
    import parity
    from oracle import metric_oracle as MO
    from test_metric_gpu import _check
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs])
    parts = eng.assess_batch([p[2] for p in probs]).split()
    for (ag, origin, ego, case), got in zip(probs, parts):
        sub = dict(case, ego=ego - np.array([origin[0], origin[1], 0, 0, 0]),
                   agents=[dict(a, pos=np.asarray(a["pos"])) for a in case["agents"]])
        # the oracle runs in the problem's own frame: the same float64 shift the batch applies
        for a, k in zip(sub["agents"], range(ag.n_agents)):
            n = int(ag.n_states[k])
            a["pos"] = np.stack((ag.x[k, :n] - origin[0], ag.y[k, :n] - origin[1]), -1).astype(np.float32).astype(np.float64)
        sub["ego"] = sub["ego"].astype(np.float32).astype(np.float64)
        out = MO.evaluate_bundle(sub)
        res = {"valid": got.valid.cpu().numpy(), "summary": got.summary.cpu().numpy(),
               "flags": got.flags.cpu().numpy().astype(np.uint32)}
        _check(parity.compare_bundle(out, res, sub))


def _scene_interface(name):
    import json
    from frenetix_occlusion_b200 import replay as R
    from frenetix_occlusion_b200.interface import FOInterface
    from frenetix_occlusion_b200.scenario import scenario_from_dict
    with open(os.path.join(GOLDEN, name)) as f:
        doc = json.load(f)
    random.seed(7)
    sc = scenario_from_dict(doc["scene"])
    ego = R.OpenLoopEgo(sc)
    fo = FOInterface(sc, ego.reference_path, R.DEFAULT_VEHICLE, sc.dt, config_path=R.deployment_config(agents=doc["agents"]))
    for ts in doc["timesteps"]:
        st = ego.state(ts)
        fo.evaluate_scenario({}, st["pos"], st["orientation"], st["pos_cl"], st["v"], ts, ego.cosy)
        if fo.agent_manager.phantom_agents:
            fan = R.frenet_fan(ego.cosy, st["pos_cl"][0], st["pos_cl"][1], st["v"], dt=ego.dt, **(doc["fan"] or {}))
            return fo, fan
    raise AssertionError(f"{name}: no cycle with phantom agents")


@pytest.mark.gpu
def test_assess_interfaces_equals_each_interface(cuda_device, monkeypatch):
    import torch
    from frenetix_occlusion_b200.batch import assess_interfaces
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    pairs = [_scene_interface(n) for n in ("scene_scenario1.json", "scene_scenario2.json", "scene_scenario3.json",
                                           "scene_parked_car.json")]
    fos, fans = [p[0] for p in pairs], [p[1] for p in pairs]
    got = assess_interfaces(fos, fans)
    for fo, fan, g in zip(fos, fans, got):
        want = fo.assess_bundle(fan)
        torch.cuda.synchronize()
        for f in ("valid", "flags", "summary"):
            assert np.array_equal(getattr(g, f).cpu().numpy(), getattr(want, f).cpu().numpy(), equal_nan=True), f
    # configurations that one batch cannot share
    fos[1].metrics._core.engine.dt = fos[1].metrics._core.engine.dt * 2
    with pytest.raises(ValueError):
        assess_interfaces(fos, fans)
    fos[1].metrics._core.engine.dt = fos[0].metrics._core.engine.dt
    fos[2].metrics._core.engine.threshold_mask ^= 1
    with pytest.raises(ValueError):
        assess_interfaces(fos, fans)
    fos[2].metrics._core.engine.threshold_mask ^= 1
    with pytest.raises(ValueError):
        assess_interfaces(fos, [fans[0], fans[1][:, :20], fans[2], fans[3]])
    with pytest.raises(ValueError):
        assess_interfaces(fos, fans[:3])
