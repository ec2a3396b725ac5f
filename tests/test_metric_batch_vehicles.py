"""Batches of independent planning problems with one ego vehicle per problem (fo_agents_pack_batch_vehicles,
fo_metric_batch_vehicles, fo_metric_batch_detail_vehicles, MetricEngine.set_agent_batch(vehicles=...), and
batch.assess_interfaces / prefetch_interfaces over interfaces with different vehicle_params).  The CPU part checks the
argument validation (before any CUDA call); the GPU part checks that every problem of a mixed-fleet batch gets exactly
what the single-problem path gives it with its own vehicle."""
import ctypes as C
import json
import os
import random
import types

import numpy as np
import pytest

from conftest import GOLDEN
from test_metric_batch import _batch_args, _problems
from test_metric_batch_detail import SCENES, _assert_same_assessments, _trajectories

FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2

# four vehicle classes of a mixed fleet; every problem jitters its class's dimensions
VEHICLE_CLASSES = (
    {"length": 3.6, "width": 1.6, "mass": 900.0, "wb_rear_axle": 1.1, "a_max": 9.5},        # compact
    None,                                                                                    # synthetic.VEHICLE (BMW 320i)
    {"length": 5.9, "width": 2.0, "mass": 2500.0, "wb_rear_axle": 1.8, "a_max": 8.0},       # van
    {"length": 12.0, "width": 2.55, "mass": 18000.0, "wb_rear_axle": 3.9, "a_max": 6.0},    # truck
)


def _fleet(n, seed):
    """n vehicles of the four classes in turn, each dimension jittered by up to 4 % (float32 values, all distinct)."""
    from frenetix_occlusion_b200 import synthetic as S
    rng = np.random.default_rng(seed)
    out = []
    for p in range(n):
        base = VEHICLE_CLASSES[p % 4] or S.VEHICLE
        out.append({k: float(np.float32(v * rng.uniform(0.96, 1.04))) for k, v in base.items()})
    keys = {tuple(v.values()) for v in out}
    assert len(keys) == n
    return out


def _mixed(seed, T, a_set=(0, 1, 3, 16, 17, 33, 300), n_set=(0, 1, 64, 500), n_problems=14, metrics=None,
           thresholds=None, varied=False):
    """Problems of test_metric_batch._problems (every agent count with every trajectory count of its residue) and one
    vehicle each."""
    probs = _problems(seed, T, n_problems=n_problems, a_set=list(a_set), n_set=list(n_set), metrics=metrics,
                      thresholds=thresholds, varied=varied)
    return probs, _fleet(len(probs), seed)


def _engine(case, vehicle=None):
    from frenetix_occlusion_b200.engine import MetricEngine
    return MetricEngine(vehicle or case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])


def _assert_equal(g, w, what):
    g, w = g.cpu().numpy(), w.cpu().numpy()
    assert g.shape == w.shape, (what, g.shape, w.shape)
    assert np.array_equal(g, w, equal_nan=True), what
    if g.dtype.kind == "f":
        assert np.array_equal(np.isnan(g), np.isnan(w)), what


def _assert_fleet_batch_equals_single(probs, fleet, want_pair=False, want_step=False):
    import torch
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet)
    parts = eng.assess_batch([p[2] for p in probs], want_pair=want_pair, want_step=want_step).split()
    fields = ("valid", "flags", "summary") + (("pair",) if want_pair else ()) + (("step",) if want_step else ())
    for i, ((ag, origin, ego, case), veh, got) in enumerate(zip(probs, fleet, parts)):
        if not len(ego):
            assert got.valid.numel() == 0
            continue
        single = _engine(case, veh)
        single.set_agents(ag, origin=origin)
        want = single.assess(ego, want_pair=want_pair, want_step=want_step)
        torch.cuda.synchronize()
        for f in fields:
            _assert_equal(getattr(got, f), getattr(want, f), (i, f, ag.n_agents, len(ego)))


# ---------------------------------------------------------------------------------------------------- CPU
def test_vehicle_entry_points_reject_null_vehicles_without_device():
    from frenetix_occlusion_b200 import _lib as L
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    assert L.lib.fo_metric_batch_vehicles(C.byref(a), None, None) == FO_ERR_INVALID_ARG
    assert b"fo_metric_batch_vehicles" in L.lib.fo_last_error()
    a.common.pair = 1 << 24
    assert L.lib.fo_metric_batch_detail_vehicles(C.byref(a), None, None) == FO_ERR_INVALID_ARG
    assert b"fo_metric_batch_detail_vehicles" in L.lib.fo_last_error()
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = 4, 31
    pr = (L.FoBatchProblem * 2)()
    pr[0].n_agents, pr[0].t_stride, pr[1].n_agents, pr[1].t_stride, pr[1].table_offset = 2, 31, 2, 31, 8192
    assert L.lib.fo_agents_pack_batch_vehicles(C.byref(raw), 2, pr, None, C.c_void_p(1 << 20), 1 << 16, None) \
        == FO_ERR_INVALID_ARG
    assert b"fo_agents_pack_batch_vehicles" in L.lib.fo_last_error()
    # no problems: nothing is read, as in the shared-vehicle calls
    assert L.lib.fo_metric_batch_vehicles(C.byref(_batch_args(L, [], 0)), None, None) == 0
    raw.n_agents = 0
    assert L.lib.fo_agents_pack_batch_vehicles(C.byref(raw), 0, None, None, None, 0, None) == 0


def _malformed_summary_cases(L):
    """(name, args) of every malformed descriptor case of test_batch_argument_validation_without_device."""
    cases = [("n_problems < 0", _batch_args(L, [], 0)), ("problems NULL", _batch_args(L, [(0, 4, 2, 31, 0)], 4))]
    cases[0][1].n_problems = -1
    cases[1][1].problems = None
    for name, pr, n, T in (("gap", [(0, 4, 2, 31, 0), (5, 3, 2, 31, 4096)], 8, 31),
                           ("order", [(4, 3, 2, 31, 0), (0, 4, 2, 31, 4096)], 7, 31),
                           ("past n_traj", [(0, 4, 2, 31, 0), (4, 5, 2, 31, 4096)], 8, 31),
                           ("uncovered", [(0, 4, 2, 31, 0)], 6, 31),
                           ("past arena", [(0, 4, 2, 31, (1 << 20) - 64)], 4, 31),
                           ("misaligned table", [(0, 4, 2, 31, 8)], 4, 31),
                           ("no states", [(0, 4, 2, 0, 0)], 4, 31),
                           ("t_stride", [(0, 4, 2, 129, 0)], 4, 31),
                           ("T", [(0, 4, 2, 31, 0)], 4, 129)):
        cases.append((name, _batch_args(L, pr, n, T)))
    for name, field in (("pair", "pair"), ("step", "step"), ("peers", "n_peers"), ("valid", "valid")):
        a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
        setattr(a.common, field, {"pair": a.common.ego, "step": a.common.ego, "n_peers": 1, "valid": None}[field])
        cases.append((name, a))
    return cases


def _malformed_detail_cases(L):
    """(name, args) of every malformed descriptor case of test_batch_detail_argument_validation_without_device."""
    def args(problems, n_traj, T=31, pair=1 << 24, step=None):
        a = _batch_args(L, problems, n_traj, T)
        a.common.agent_table = 1 << 20
        a.common.pair, a.common.step = pair, step
        return a
    ok = [(0, 4, 2, 31, 0)]
    cases = [("no detail", args(ok, 4, pair=None)), ("pair align", args(ok, 4, pair=(1 << 24) + 8)),
             ("step align", args(ok, 4, pair=None, step=(1 << 24) + 2))]
    a = args(ok, 4)
    a.common.n_peers = 1
    cases.append(("peers", a))
    a = args([], 0)
    a.n_problems = -1
    cases.append(("n_problems < 0", a))
    a = args(ok, 4)
    a.problems = None
    cases.append(("problems NULL", a))
    for step in (None, 1 << 26):
        for name, pr, n, T in (("gap", [(0, 4, 2, 31, 0), (5, 3, 2, 31, 4096)], 8, 31),
                               ("order", [(4, 3, 2, 31, 0), (0, 4, 2, 31, 4096)], 7, 31),
                               ("past n_traj", [(0, 4, 2, 31, 0), (4, 5, 2, 31, 4096)], 8, 31),
                               ("uncovered", ok, 6, 31), ("past arena", [(0, 4, 2, 31, (1 << 20) - 64)], 4, 31),
                               ("misaligned table", [(0, 4, 2, 31, 8)], 4, 31), ("no states", [(0, 4, 2, 0, 0)], 4, 31),
                               ("t_stride", [(0, 4, 2, 129, 0)], 4, 31), ("T", ok, 4, 129)):
            cases.append((f"{name} step={step}", args(pr, n, T, step=step)))
    for name, field, value in (("arena align", "agent_table", (1 << 20) + 8), ("be without ttc", "metric_mask", 1 << 4),
                               ("valid", "valid", None), ("summary align", "summary", (1 << 24) + 4)):
        a = args(ok, 4)
        setattr(a.common, field, value)
        cases.append((name, a))
    return cases


def test_vehicle_entry_points_validate_like_their_shared_vehicle_counterparts_without_device():
    from frenetix_occlusion_b200 import _lib as L
    fleet = (L.FoVehicle * 8)(*[L.FoVehicle(4.5, 1.6, 1200.0, 1.4, 10.0) for _ in range(8)])
    for fn, cases in (("fo_metric_batch", _malformed_summary_cases(L)),
                      ("fo_metric_batch_detail", _malformed_detail_cases(L))):
        for name, a in cases:
            old = getattr(L.lib, fn)(C.byref(a), None)
            new = getattr(L.lib, fn + "_vehicles")(C.byref(a), fleet, None)
            assert old != 0 and new == old, (fn, name, old, new)
            assert (fn + "_vehicles").encode() in L.lib.fo_last_error(), (fn, name)
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = 3, 31
    pr = (L.FoBatchProblem * 2)()
    pr[0].n_agents, pr[0].t_stride, pr[1].n_agents, pr[1].t_stride, pr[1].table_offset = 2, 31, 2, 31, 8192
    arena = C.c_void_p(1 << 20)
    for n_agents, arena_bytes, r in ((3, 1 << 16, raw), (4, 8192, raw), (4, 1 << 16, raw), (4, 1 << 16, None)):
        raw.n_agents = n_agents
        rp = C.byref(r) if r is not None else None
        old = L.lib.fo_agents_pack_batch(rp, 2, pr, fleet, arena, arena_bytes, None)
        new = L.lib.fo_agents_pack_batch_vehicles(rp, 2, pr, fleet, arena, arena_bytes, None)
        assert old == FO_ERR_INVALID_ARG and new == old, (n_agents, arena_bytes, old, new)


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("warps", [1, 4])
def test_fleet_batch_equals_single_problem_path(T, warps, cuda_device, monkeypatch):
    """W = 1 mixes the window-filter class (>= 17 agents) and the team class in one batch."""
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    probs, fleet = _mixed(T + 200, T)
    assert {p[0].n_agents for p in probs} == {0, 1, 3, 16, 17, 33, 300} and {len(p[2]) for p in probs} == {0, 1, 64, 500}
    _assert_fleet_batch_equals_single(probs, fleet)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("detail", ["pair", "step", "both"])
def test_fleet_detail_batch_equals_single_problem_path(T, detail, cuda_device):
    probs, fleet = _mixed(T + 300, T)
    _assert_fleet_batch_equals_single(probs, fleet, detail != "step", detail != "pair")


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", [None, "default", ["dce", "ttc", "wttc"], ["ttc", "be", "hr", "cp"]])
@pytest.mark.parametrize("armed", [False, True])
@pytest.mark.parametrize("detail", [False, True])
def test_fleet_batch_equals_single_problem_path_metrics_and_thresholds(metrics, armed, detail, cuda_device,
                                                                       monkeypatch):
    """None is all seven metrics with BE; the last set runs BE through the kernels without a compile-time metric set.
    Armed dce / ttc / be thresholds run the float64 rounding-tie variants."""
    from frenetix_occlusion_b200 import synthetic as S
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    m = S.DEFAULT_METRICS if metrics == "default" else metrics
    thr = dict(S.DEFAULT_THRESHOLDS, dce=0.5, ttc=1.5, be=0.8) if armed else None
    probs, fleet = _mixed(37 + armed, 31, metrics=m, thresholds=thr, n_set=(0, 1, 64, 200))
    _assert_fleet_batch_equals_single(probs, fleet, detail, detail)


@pytest.mark.gpu
def test_fleet_tables_are_byte_identical_to_single_packs(cuda_device):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    probs, fleet = _mixed(41, 51, n_set=(1,))
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet)
    arena = eng._batch["arena"]
    for p, ((ag, origin, _, case), veh) in enumerate(zip(probs, fleet)):
        if ag.n_agents == 0:
            continue
        single = _engine(case, veh)
        single.set_agents(ag, origin=origin)
        off = eng._batch["problems"][p].table_offset
        n = L.lib.fo_agent_table_bytes(ag.n_agents, ag.t_stride)
        torch.cuda.synchronize()
        assert torch.equal(arena[off:off + n], single._table[:n]), p


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_the_vehicle_changes_the_result(detail, cuda_device, monkeypatch):
    """One problem, assessed in one batch with a compact and with a truck, gets different summaries: a kernel that read
    the shared vehicle would give both the same.  The synthetic scenes collide at the first step, so min_dce is checked
    on a copy of the bundle moved 25 m sideways."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    probs, _ = _mixed(43, 31, a_set=(8, 40), n_set=(200,), n_problems=2)
    compact, truck = _fleet(4, 43)[0], _fleet(4, 43)[3]
    for ag, origin, ego, case in probs:
        far = ego.copy()
        far[..., 1] += 25.0
        eng = _engine(case)
        eng.set_agent_batch([ag] * 4, [origin] * 4, vehicles=[compact, truck, compact, truck])
        sa, sb, fa, fb = [r.summary.cpu().numpy() for r in
                          eng.assess_batch([ego, ego, far, far], want_pair=detail, want_step=detail).split()]
        for col in (2, 4):                   # max ego harm (mass split), max collision probability (CP ego boxes)
            assert not np.array_equal(sa[:, col], sb[:, col]), col
        assert np.any(np.isfinite(fa[:, 6]) & (fa[:, 6] > 0))
        assert not np.array_equal(fa[:, 6], fb[:, 6])    # min_dce (ego box)


@pytest.mark.gpu
def test_every_problem_of_a_fleet_batch_matches_the_oracle(cuda_device, monkeypatch):
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    _assert_every_fleet_problem_matches_the_oracle(*_mixed(47, 31, a_set=(0, 3, 17, 40), n_set=(60, 25, 80, 30), n_problems=8))


@pytest.mark.gpu
def test_every_problem_of_a_fleet_batch_matches_the_oracle_on_varied_agents(cuda_device, monkeypatch):
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    _assert_every_fleet_problem_matches_the_oracle(*_mixed(48, 51, a_set=(0, 5, 17, 40), n_set=(60, 25, 80, 30),
                                                           n_problems=8, varied=True))


def _assert_every_fleet_problem_matches_the_oracle(probs, fleet):
    import parity
    from oracle import metric_oracle as MO
    from test_metric_gpu import _check
    for detail in (False, True):
        eng = _engine(probs[0][3])
        eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet)
        parts = eng.assess_batch([p[2] for p in probs], want_pair=detail, want_step=detail).split()
        for (ag, origin, ego, case), veh, got in zip(probs, fleet, parts):
            sub = dict(case, vehicle=dict(veh), ego=ego - np.array([origin[0], origin[1], 0, 0, 0]),
                       agents=[dict(a, pos=np.asarray(a["pos"])) for a in case["agents"]])
            # the oracle runs in the problem's own frame: the same float64 shift the batch applies
            for a, k in zip(sub["agents"], range(ag.n_agents)):
                n = int(ag.n_states[k])
                a["pos"] = np.stack((ag.x[k, :n] - origin[0], ag.y[k, :n] - origin[1]), -1).astype(np.float32).astype(np.float64)
            sub["ego"] = sub["ego"].astype(np.float32).astype(np.float64)
            out = MO.evaluate_bundle(sub)
            res = {"valid": got.valid.cpu().numpy(), "summary": got.summary.cpu().numpy(),
                   "flags": got.flags.cpu().numpy().astype(np.uint32)}
            if detail:
                res["pair"], res["step"] = got.pair.cpu().numpy(), got.step.cpu().numpy()
            _check(parity.compare_bundle(out, res, sub))


# ---- interfaces with different vehicle_params ------------------------------------------------------------------
def _scene_interface_with(name, vehicle):
    """test_metric_batch._scene_interface with the interface's vehicle_params = vehicle."""
    from frenetix_occlusion_b200 import replay as R
    from frenetix_occlusion_b200.interface import FOInterface
    from frenetix_occlusion_b200.scenario import scenario_from_dict
    with open(os.path.join(GOLDEN, name)) as f:
        doc = json.load(f)
    random.seed(7)
    sc = scenario_from_dict(doc["scene"])
    ego = R.OpenLoopEgo(sc)
    fo = FOInterface(sc, ego.reference_path, types.SimpleNamespace(**vehicle), sc.dt,
                     config_path=R.deployment_config(agents=doc["agents"]))
    for ts in doc["timesteps"]:
        st = ego.state(ts)
        fo.evaluate_scenario({}, st["pos"], st["orientation"], st["pos_cl"], st["v"], ts, ego.cosy)
        if fo.agent_manager.phantom_agents:
            fan = R.frenet_fan(ego.cosy, st["pos_cl"][0], st["pos_cl"][1], st["v"], dt=ego.dt, **(doc["fan"] or {}))
            return fo, fan
    raise AssertionError(f"{name}: no cycle with phantom agents")


def _fleet_scenes():
    fleet = _fleet(len(SCENES), 53)
    pairs = [_scene_interface_with(n, v) for n, v in zip(SCENES, fleet)]
    return [p[0] for p in pairs], [p[1] for p in pairs]


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_assess_interfaces_of_a_mixed_fleet_equals_each_interface(detail, cuda_device, monkeypatch):
    import torch
    from frenetix_occlusion_b200.batch import assess_interfaces
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    fos, fans = _fleet_scenes()
    got = assess_interfaces(fos, fans, want_pair=detail, want_step=detail)
    for fo, fan, g in zip(fos, fans, got):
        want = fo.assess_bundle(fan, detail, detail)
        torch.cuda.synchronize()
        for f in ("valid", "flags", "summary") + (("pair", "step") if detail else ()):
            _assert_equal(getattr(g, f), getattr(want, f), f)


@pytest.mark.gpu
def test_prefetch_interfaces_of_a_mixed_fleet_serves_every_candidate_like_each_interface(cuda_device):
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.batch import prefetch_interfaces
    fos, fans = _fleet_scenes()
    cands = [_trajectories(f) for f in fans]
    l0 = L.lib.fo_launch_count()
    counts = prefetch_interfaces(fos, cands)
    assert L.lib.fo_launch_count() - l0 == 3            # two pack launches and one detail launch for all interfaces
    assert counts == [len(c) for c in cands]
    l0 = L.lib.fo_launch_count()
    served = [[fo.trajectory_safety_assessment(t) for t in c] for fo, c in zip(fos, cands)]
    assert L.lib.fo_launch_count() == l0, "prefetched trajectories must not launch again"
    for fo, c, s in zip(fos, cands, served):
        fo.metrics._core._fingerprint = None            # the interface's own path from scratch: sync, pack, prefetch
        assert fo.prefetch_assessments(c) == len(c)
        _assert_same_assessments(s, [fo.trajectory_safety_assessment(t) for t in c])


@pytest.mark.gpu
def test_mixed_fleet_batches_still_share_the_rest_of_the_configuration(cuda_device):
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.batch import assess_interfaces, prefetch_interfaces
    fos, fans = _fleet_scenes()
    engs = [fo.metrics._core.engine for fo in fos]
    cands = [_trajectories(f) for f in fans]

    def rejected():
        with pytest.raises(ValueError):
            assess_interfaces(fos, fans)
        with pytest.raises(ValueError):
            prefetch_interfaces(fos, cands)
    engs[1].dt *= 2
    rejected()
    engs[1].dt = engs[0].dt
    engs[2].threshold_mask ^= 1
    rejected()
    engs[2].threshold_mask ^= 1
    engs[3].metric_mask ^= L.M_BITS["wttc"]
    rejected()
    engs[3].metric_mask ^= L.M_BITS["wttc"]
    saved = L.FoHarmCoeffs.from_buffer_copy(engs[1].harm)
    engs[1].harm.rs_speed *= 1.5
    rejected()
    engs[1].harm = saved
    with pytest.raises(ValueError):
        assess_interfaces(fos, [fans[0], fans[1][:, :20], fans[2], fans[3]])
    assess_interfaces(fos, fans)                        # the vehicles differ, everything else agrees
