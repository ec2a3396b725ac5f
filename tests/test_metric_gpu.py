"""Parity of the CUDA dense metric core (through the C ABI) against the float64 oracle and the
reference-generated golden vectors.  Needs a GPU: run with ``-m gpu`` on the B200 box."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_files
from frenetix_occlusion_b200 import synthetic as S
from oracle import metric_oracle as MO
from oracle.compare import compare_results
import parity

pytestmark = pytest.mark.gpu


def _check(rep, max_tie_rate=0.005):
    """Documented exact-threshold ties (DESIGN.md 2) are bounded at 0.5 % of the pairs -- the observed level is 0.14 %,
    all of them risk-argmax indices of two float32 products equal within rounding."""
    assert not rep["fail"], "\n".join(rep["fail"])
    n_ties = sum(rep["ties"].values())
    assert n_ties <= max(3, max_tie_rate * rep["n_pairs"]), rep["ties"]


@pytest.mark.parametrize("fname", golden_files("metric_"))
def test_cuda_matches_oracle_on_golden_cases(fname, cuda_device):
    case, reference, order = MO.load_case_json(os.path.join(GOLDEN, fname))
    out = MO.evaluate_bundle(case)
    res, eng = parity.run_gpu(case)
    assert eng.order == order
    _check(parity.compare_bundle(out, res, case))


@pytest.mark.parametrize("fname", ["metric_kat_pedestrian.json", "metric_closed_form.json", "metric_ragged_lengths.json"])
def test_cuda_matches_reference_dicts_directly(fname, cuda_device):
    """The drop-in ``Metric.evaluate_metrics`` against the reference's own result dicts."""
    from frenetix_occlusion_b200.metrics.metric import Metric
    from oracle.ref_runner import TrajectoryStub
    from oracle import ref_runner
    import types
    case, reference, order = MO.load_case_json(os.path.join(GOLDEN, fname))
    am = _agent_manager_from_case(case)
    vp = types.SimpleNamespace(**case["vehicle"])
    metric = Metric({"activated_metrics": list(case["activated_metrics"]), "metric_thresholds": dict(case["thresholds"])},
                    vp, am)
    assert list(metric.metrics.keys()) == order
    for n, ref in enumerate(reference):
        if ref["safety_check"] is None:
            with pytest.raises(ValueError):
                metric.evaluate_metrics(TrajectoryStub(case["ego"][n]))
            continue
        results, ok = metric.evaluate_metrics(TrajectoryStub(case["ego"][n]))
        problems = compare_results(ref["results"], results, rtol=1e-4, atol=2e-6)
        assert not problems, f"{fname}[{n}]:\n" + "\n".join(problems[:10])
        assert ok == ref["safety_check"]


def _agent_manager_from_case(case):
    import types
    am = types.SimpleNamespace(dt=case["dt"], visualization=None, phantom_agents=[], predictions={})
    for k, ag in enumerate(case["agents"]):
        agent = types.SimpleNamespace(agent_id=10000 + k, agent_type=ag["agent_type"],
                                      shape=types.SimpleNamespace(length=ag["length"], width=ag["width"]))
        am.phantom_agents.append(agent)
        var = np.asarray(ag["var"])
        am.predictions[int(str(10000 + k) + "0")] = {
            "orientation_list": np.asarray(ag["yaw"]), "v_list": np.asarray(ag["v"]),
            "pos_list": np.asarray(ag["pos"]).reshape(-1, 2),
            "shape": {"length": ag["buf_length"], "width": ag["buf_width"]},
            "cov_list": np.array([[[v, 0.0], [0.0, v]] for v in var])}
    am.agent_by_prediction_id = lambda pid: next(a for a in am.phantom_agents if a.agent_id == int(str(pid)[:5]))
    return am


@pytest.mark.parametrize("seed,n,a,t", [(1, 64, 16, 31), (2, 50, 12, 51), (3, 200, 32, 31), (4, 33, 5, 2), (5, 40, 9, 97)])
def test_cuda_matches_oracle_on_random_bundles(seed, n, a, t, cuda_device):
    case = S.make_case(n, a, t, seed=seed)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case)
    _check(parity.compare_bundle(out, res, case))


def test_latency_config_parity(cuda_device):
    """BASELINE config C-lat (1k x 32 x 30 steps), all seven metrics, full detail compared."""
    case = S.make_case(1000, 32, 31)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case)
    rep = parity.compare_bundle(out, res, case)
    _check(rep)


def test_summary_kernel_equals_detail_kernel(cuda_device):
    """The summary kernel (bench / planner path) against the detail kernel at a size the CPU
    oracle would need minutes for: identical masks/flags/discrete values, floats to 1e-5."""
    assert_summary_equals_detail(S.make_case(3000, 300, 51, seed=9))      # > 256 agents: exercises agent tiling


def assert_summary_equals_detail(case):
    res_d, _ = parity.run_gpu(case, want_pair=True, want_step=True)
    res_s, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    # FO_F_BE_RANGE is a float32 comparison (re-timed path length vs original path length); the two
    # kernels sum the series differently, so a handful of near-equal cases may flip (documented tie)
    same = res_d["flags"] == res_s["flags"]
    assert (~same).sum() <= max(2, 0.005 * len(same)), int((~same).sum())
    assert np.array_equal(res_d["valid"][same], res_s["valid"][same])
    ok = ((res_d["flags"] & 1) == 0) & same
    # wttc: discrete.  min dce: the detail kernel re-rounds float32 rounding ties from a float64 evaluation
    # (np.round(d, 3) next to a x.xxx5 boundary), the summary kernel does not: the last digit may differ on a few
    assert np.array_equal(res_d["summary"][:, 7], res_s["summary"][:, 7])
    dd = np.abs(res_d["summary"][:, 6] - res_s["summary"][:, 6])
    assert (dd > 0).sum() <= max(2, 0.005 * len(dd)) and np.all(dd[dd > 0] < 0.0011)
    be_same = res_d["summary"][ok, 9] == res_s["summary"][ok, 9]     # bisection ties (one probe flips)
    assert (~be_same).sum() <= max(2, 0.005 * ok.sum()), int((~be_same).sum())
    # the summary kernels use the 18-instruction erfc (4e-6 relative in float32), the detail kernel CUDA's erfcf
    for col in range(6):
        np.testing.assert_allclose(res_s["summary"][:, col], res_d["summary"][:, col], rtol=3e-5, atol=1e-7)
    ok = (res_d["flags"] & 1) == 0
    # and the summary is the reduction of the per-pair detail
    p = res_d["pair"]
    assert np.array_equal(res_d["summary"][:, 6], p[..., 0].min(1))
    assert np.array_equal(res_d["summary"][ok, 8], p[ok][..., 10].max(1))
    for col_s, col_p in ((0, 2), (1, 3), (2, 6), (3, 7), (4, 8), (5, 5)):
        assert np.array_equal(res_d["summary"][:, col_s], p[..., col_p].max(1))


@pytest.mark.parametrize("seed,n,a,t", [(31, 500, 32, 31), (32, 200, 40, 51), (33, 100, 7, 2), (34, 64, 300, 31)])
def test_summary_kernel_matches_oracle(seed, n, a, t, cuda_device):
    case = S.make_case(n, a, t, seed=seed)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    _check(parity.compare_bundle(out, res, case))


@pytest.mark.parametrize("seed,n,a,t,metrics", [(35, 300, 32, 31, None), (36, 120, 300, 51, None), (37, 200, 20, 12, None),
                                                (38, 150, 64, 97, None), (39, 200, 40, 31, ["hr", "cp"]),
                                                (40, 200, 40, 31, ["dce", "ttc", "wttc"]),
                                                (41, 100, 17, 9, None), (42, 100, 33, 8, None), (43, 60, 64, 2, None),
                                                (44, 40, 32, 128, None)])
def test_window_filter_shape_matches_oracle(seed, n, a, t, metrics, cuda_device, monkeypatch):
    """One warp per trajectory and >= 17 agents is the throughput shape with the (agent, 8-step window) filter in
    front of the per-step loop; bundles this small normally take the multi-warp shape, so force it."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    case = S.make_case(n, a, t, seed=seed, activated_metrics=metrics)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    _check(parity.compare_bundle(out, res, case))


@pytest.mark.parametrize("metrics,thr", [
    (["hr", "ttc", "ttce", "dce", "wttc", "cp"], {"harm": 0.1, "risk": 1, "be": None, "cp": None, "ttc": None, "dce": None}),
    (["dce", "ttc"], {"harm": None, "risk": None, "be": None, "cp": None, "ttc": 1.2, "dce": 0.75}),
    (["cp"], {"harm": 0.1, "risk": 1, "be": None, "cp": 0.1, "ttc": None, "dce": None}),
    (["hr"], {"harm": 0.2, "risk": 0.02, "be": None, "cp": 0.15, "ttc": None, "dce": None}),
    (["be", "ttc"], {"harm": None, "risk": None, "be": 0.25, "cp": None, "ttc": None, "dce": None}),
])
def test_metric_subsets_and_thresholds(metrics, thr, cuda_device):
    """Activation subsets / armed thresholds (metric.py:50-98, 125-147) on both kernels."""
    case = S.make_case(300, 24, 31, seed=41, activated_metrics=metrics, thresholds={**thr, "wttc": None, "ttce": None})
    out = MO.evaluate_bundle(case)
    for detail in (True, False):
        res, eng = parity.run_gpu(case, want_pair=detail, want_step=detail)
        assert eng.order == out["order"]
        _check(parity.compare_bundle(out, res, case))


def test_edge_cases(cuda_device):
    # no agents -> every trajectory valid (metric.py:44-45)
    case = S.make_case(10, 0, 31)
    res, _ = parity.run_gpu(case)
    assert res["valid"].all()
    # empty bundle
    case = S.make_case(0, 4, 31)
    res, _ = parity.run_gpu(case)
    assert res["valid"].shape == (0,)
    # thresholds: translation invariance through the origin shift
    case = S.make_case(40, 8, 31, seed=21)
    res0, _ = parity.run_gpu(case)
    import copy
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    import torch
    shifted = copy.deepcopy(case)
    off = np.array([4096.0, -2048.0])     # exactly representable shift
    shifted["ego"][..., 0:2] += off
    for ag in shifted["agents"]:
        ag["pos"] = np.asarray(ag["pos"]) + off
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(shifted["agents"]), origin=off)
    r = eng.assess(shifted["ego"])
    torch.cuda.synchronize()
    assert np.array_equal(r.valid.cpu().numpy(), res0["valid"])
    sm = r.summary.cpu().numpy()
    assert np.array_equal(sm[:, 6:], res0["summary"][:, 6:], equal_nan=True)       # dce / wttc / BE: discrete
    np.testing.assert_allclose(sm[:, :6], res0["summary"][:, :6], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("seed,n,a,t", [(51, 1, 1, 31), (52, 3, 2, 31), (53, 37, 3, 31), (54, 20, 5, 51), (55, 64, 9, 31),
                                        (56, 50, 17, 31), (57, 16, 33, 31), (58, 8, 257, 31), (59, 6, 600, 16),
                                        (60, 5, 40, 128), (61, 1500, 32, 31), (62, 9000, 8, 31)])
def test_summary_kernel_shapes(seed, n, a, t, cuda_device):
    """Lane-group boundaries (agents 1..33 -> 1..32 lanes per slice), more than one 256-agent tile, the maximum
    number of states (FO_MAX_STATES = 128), a single trajectory, and bundles on both sides of the one-wave limit
    (team width 1..8)."""
    case = S.make_case(n, a, t, seed=seed)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    _check(parity.compare_bundle(out, res, case))


def test_ragged_agent_lengths_summary(cuda_device):
    """Predictions shorter and longer than the ego horizon (dce.py:87-88, collision_probability.py:49-51,
    harm_model.py:67-70) through the summary kernel."""
    case = S.make_case(120, 12, 31, seed=71, agent_states=51)
    for k, ag in enumerate(case["agents"]):
        keep = [51, 31, 30, 12, 2, 1][k % 6]
        for key in ("pos", "yaw", "v", "var"):
            ag[key] = np.asarray(ag[key])[:keep]
    out = MO.evaluate_bundle(case)
    for detail in (False, True):
        res, _ = parity.run_gpu(case, want_pair=detail, want_step=detail)
        _check(parity.compare_bundle(out, res, case))


def test_ragged_agent_lengths_window_filter(cuda_device, monkeypatch):
    """The same ragged predictions through the one-warp shape: windows that an agent only partly has, or does not
    have at all, must neither be evaluated nor hide a step."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    case = S.make_case(150, 36, 31, seed=72, agent_states=51)
    for k, ag in enumerate(case["agents"]):
        keep = [51, 31, 30, 17, 16, 9, 8, 2, 1][k % 9]
        for key in ("pos", "yaw", "v", "var"):
            ag[key] = np.asarray(ag[key])[:keep]
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    _check(parity.compare_bundle(out, res, case))


@pytest.mark.parametrize("thr", [{"dce": 0.75, "ttc": 1.2}, {"dce": 0.3, "ttc": None}, {"dce": None, "ttc": 2.0}])
def test_armed_distance_thresholds_on_the_window_filter_shape(thr, cuda_device, monkeypatch):
    """dce / ttc thresholds armed on the throughput shape (one warp per trajectory, window filter): the clauses compare
    np.round(d, 3) in float64 (dce.py:79, ttc.py:43, metric.py:85-98), so the summary kernel runs its float64 tie
    re-rounding variant and the mask must equal the oracle's bit for bit -- no tie allowance for dce rounding."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    thresholds = {"harm": None, "risk": None, "be": None, "cp": None, "wttc": None, "ttce": None, **thr}
    case = S.make_case(4000, 48, 51, seed=93, thresholds=thresholds)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    rep = parity.compare_bundle(out, res, case)
    assert not rep["fail"], "\n".join(rep["fail"])
    ok = ~out["be_error"] & ((res["flags"] & 1) == 0)
    assert np.array_equal(res["valid"].astype(bool)[ok], out["valid"][ok])
    assert np.array_equal(np.round(res["summary"][ok, 6].astype(np.float64), 3), out["dce"].min(1)[ok])
    assert 0 < out["valid"].sum() < len(out["valid"])          # the clauses really decide something here


def test_exact_dce_switch_matches_detail_kernel(cuda_device, monkeypatch):
    """FO_EXACT_DCE=1 turns the float64 tie re-rounding on without any armed distance threshold: min_dce of the
    summary kernel then equals the detail kernel's on every trajectory."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    monkeypatch.setenv("FO_EXACT_DCE", "1")
    case = S.make_case(3000, 64, 51, seed=94)
    res_d, _ = parity.run_gpu(case, want_pair=True, want_step=False)
    res_s, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    assert np.array_equal(res_d["summary"][:, 6], res_s["summary"][:, 6])
    assert np.array_equal(res_d["summary"][:, 7], res_s["summary"][:, 7])


def test_claimed_trajectories_equal_static_striding(cuda_device, monkeypatch):
    """More trajectories than resident teams: the summary kernel hands trajectories out through a device counter
    (zeroed in-stream per launch).  Same bits as static striding, eagerly and when the launch -- with its counter
    reset -- is replayed from a CUDA graph."""
    import torch
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    case = S.make_case(40000, 6, 31, seed=83)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    ego = torch.from_numpy(np.ascontiguousarray(case["ego"], dtype=np.float32)).cuda()
    monkeypatch.setenv("FO_STATIC_STRIDE", "1")
    ref = eng.assess(ego)
    torch.cuda.synchronize()
    ref = [x.cpu().numpy().copy() for x in (ref.valid, ref.summary, ref.flags)]
    monkeypatch.delenv("FO_STATIC_STRIDE")
    for _ in range(3):
        r = eng.assess(ego)
        torch.cuda.synchronize()
        for a, b in zip(ref, (r.valid, r.summary, r.flags)):
            assert np.array_equal(a, b.cpu().numpy(), equal_nan=True)
    g, out = eng.capture(ego)
    for _ in range(3):
        out.summary.fill_(-1.0)
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(ref, (out.valid, out.summary, out.flags)):
            assert np.array_equal(a, b.cpu().numpy(), equal_nan=True)


@pytest.mark.parametrize("n,a,t,detail", [(200, 12, 31, True), (60000, 4, 31, False), (7, 0, 31, False)])
def test_host_buffer_entry_point(n, a, t, detail, cuda_device):
    """fo_metric_bundle_host (the C-ABI call a non-torch embedder makes: host pointers in, host pointers out) equals
    the device-resident path -- small bundle with detail outputs, a bundle large enough for the chunked H2D/compute
    pipeline, and no agents."""
    import ctypes as C
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import AgentSet, BundleResult, MetricEngine
    case = S.make_case(n, a, t, seed=81)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    ag = AgentSet.from_case(case["agents"])
    eng.set_agents(ag)
    ego = np.ascontiguousarray(case["ego"], dtype=np.float32)
    r = eng.assess(torch.from_numpy(ego).cuda(), want_pair=detail, want_step=detail)
    torch.cuda.synchronize()
    f32 = lambda x: np.ascontiguousarray(x, dtype=np.float32)  # noqa: E731
    keep = [f32(ag.x), f32(ag.y), f32(ag.yaw), f32(ag.v), f32(ag.var_x), f32(ag.var_y),
            np.ascontiguousarray(ag.n_states, dtype=np.int32), np.ascontiguousarray(ag.kind, dtype=np.int32),
            f32(ag.length), f32(ag.width), f32(ag.buf_length), f32(ag.buf_width)]
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = ag.n_agents, max(ag.t_stride, 0)
    (raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y, raw.n_states, raw.kind, raw.length, raw.width, raw.buf_length,
     raw.buf_width) = [x.ctypes.data if x.size else None for x in keep]
    out = BundleResult(torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty((n, L.FO_SUMMARY_K), device="cuda"),
                       torch.empty(n, dtype=torch.int32, device="cuda"))
    prm = eng._args(torch.from_numpy(ego).cuda(), out)
    valid, summ, flags = np.empty(n, np.uint8), np.empty((n, L.FO_SUMMARY_K), np.float32), np.empty(n, np.uint32)
    pair = np.empty((n, a, L.FO_PAIR_K), np.float32) if detail else None
    step = np.empty((n, a, t - 1, L.FO_STEP_K), np.float32) if detail else None
    ptr = lambda x: None if x is None else C.c_void_p(x.ctypes.data)  # noqa: E731
    L.check(L.lib.fo_metric_bundle_host(ptr(ego), n, t, C.byref(raw), C.byref(prm), ptr(valid), ptr(summ), ptr(flags),
                                        ptr(pair), ptr(step)), "fo_metric_bundle_host")
    assert np.array_equal(valid, r.valid.cpu().numpy())
    assert np.array_equal(flags, r.flags.cpu().numpy().astype(np.uint32))
    assert np.array_equal(summ, r.summary.cpu().numpy(), equal_nan=True)
    if detail:
        assert np.array_equal(pair, r.pair.cpu().numpy(), equal_nan=True)
        assert np.array_equal(step, r.step.cpu().numpy(), equal_nan=True)


def test_full_size_sweep_properties(cuda_device):
    """BASELINE.json configs[3] at FULL size (1,000,000 trajectories x 256 agents x 50 steps, all seven metrics):
    size-independent properties of the summary path plus an oracle spot check.
    * idempotence: two passes give bit-identical outputs;
    * sharding invariance: evaluating the two halves separately equals the whole (the multi-GPU split);
    * agent-order invariance: every per-trajectory output is an order-independent min / max over agents, so a
      permuted agent table gives bit-identical masks, discrete outputs and maxima;
    * 96 trajectories drawn from the million agree with the float64 oracle."""
    import torch
    import bench
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    wl = dict(S.C_SWEEP)
    N, A, T = wl["n_traj"], wl["n_agents"], wl["n_states"]
    case = bench.make_case(wl, N)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    ego = torch.from_numpy(case["ego"]).cuda()

    def run(e, bundle):
        r = e.assess(bundle)
        torch.cuda.synchronize()
        return r.valid.clone(), r.summary.clone(), r.flags.clone()

    v0, s0, f0 = run(eng, ego)
    v1, s1, f1 = run(eng, ego)
    assert torch.equal(v0, v1) and torch.equal(f0, f1) and torch.equal(s0.view(torch.int32), s1.view(torch.int32))
    half = N // 2
    va, sa, fa = run(eng, ego[:half])
    vb, sb, fb = run(eng, ego[half:])
    assert torch.equal(torch.cat((va, vb)), v0) and torch.equal(torch.cat((fa, fb)), f0)
    assert torch.equal(torch.cat((sa, sb)).view(torch.int32), s0.view(torch.int32))
    perm = np.random.default_rng(3).permutation(A)
    eng_p = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng_p.set_agents(AgentSet.from_case([case["agents"][j] for j in perm]))
    vp, sp, fp = run(eng_p, ego)
    assert torch.equal(vp, v0) and torch.equal(fp, f0)
    assert torch.equal(sp.view(torch.int32), s0.view(torch.int32))
    assert float(s0[:, 4].max()) > 0.05 and float(s0[:, 6].min()) == 0.0     # the sweep is dense: CP and collisions occur
    # oracle spot check
    idx = np.sort(np.random.default_rng(4).choice(N, 96, replace=False))
    sub = dict(case)
    sub["ego"] = case["ego"][idx].astype(np.float64)
    out = MO.evaluate_bundle(sub)
    res = {"valid": v0.cpu().numpy()[idx], "summary": s0.cpu().numpy()[idx], "flags": f0.cpu().numpy()[idx].astype(np.uint32),
           "pair": None, "step": None}
    _check(parity.compare_bundle(out, res, sub))


def test_per_trajectory_results_are_never_reused_across_trajectories(cuda_device):
    """Regression: the per-trajectory result cache must not key on id() of freed objects.  Freshly built trajectory
    objects that are dropped right after their call (CPython then reuses their addresses) and whose ``cartesian.x``
    is a new array per access (pybind-style) must each get their own results; an in-place edit must be seen too."""
    import types
    from frenetix_occlusion_b200.metrics.metric import Metric
    case = S.make_case(24, 6, 31, seed=21)
    out = MO.evaluate_bundle(case)
    am = _agent_manager_from_case(case)
    vp = types.SimpleNamespace(**case["vehicle"])
    metric = Metric({"activated_metrics": list(case["activated_metrics"]), "metric_thresholds": dict(case["thresholds"])}, vp, am)

    class Cart:
        def __init__(self, arr):
            self._a = arr
        x = property(lambda self: np.array(self._a[:, 0]))
        y = property(lambda self: np.array(self._a[:, 1]))
        theta = property(lambda self: np.array(self._a[:, 2]))
        v = property(lambda self: np.array(self._a[:, 3]))
        a = property(lambda self: np.array(self._a[:, 4]))

    pids = list(am.predictions.keys())
    for n in range(24):
        tr = types.SimpleNamespace(cartesian=Cart(np.asarray(case["ego"][n], dtype=np.float64)))
        results, ok = metric.evaluate_metrics(tr)
        got = np.array([results["dce"][p]["dce"] for p in pids])
        assert np.array_equal(got, out["dce"][n]), n
        assert ok == bool(out["valid"][n])
        del tr, results
    # in-place mutation of one object between two calls
    arr = np.array(case["ego"][0], dtype=np.float64)
    tr = types.SimpleNamespace(cartesian=Cart(arr))
    r0, _ = metric.evaluate_metrics(tr)
    arr[:] = case["ego"][5]
    r1, _ = metric.evaluate_metrics(tr)
    assert np.array_equal(np.array([r1["dce"][p]["dce"] for p in pids]), out["dce"][5])
    # prefetch: one launch for all candidates, the per-trajectory calls answer from the host copy with equal dicts
    trs = [types.SimpleNamespace(cartesian=Cart(np.asarray(case["ego"][n], dtype=np.float64))) for n in range(24)]
    direct = [metric.evaluate_metrics(t) for t in trs]
    from frenetix_occlusion_b200 import _lib as L
    metric.prefetch(trs)
    l0 = L.lib.fo_launch_count()
    served = [metric.evaluate_metrics(t) for t in trs]
    assert L.lib.fo_launch_count() == l0, "prefetched trajectories must not launch again"
    for (ra, oka), (rb, okb) in zip(direct, served):
        assert oka == okb and not compare_results(ra, rb, rtol=0, atol=0)
