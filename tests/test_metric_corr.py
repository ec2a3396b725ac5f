"""Predictions with full 2x2 covariances: the collision probability of the dense metric core with correlated
covariances (fo_agents_pack_corr / fo_metric_bundle_corr, MetricEngine with AgentSet.cov_xy).

CPU: the oracle's rectangle mass against a 1-D quadrature and scipy, AgentSet validation, C-ABI argument checks and the
code-size budgets of the new kernels.  GPU (-m gpu): parity with the float64 oracle on the summary and detail kernels,
the drop-in Metric protocol, the correlated table with zero correlation against the diagonal path, CUDA-graph capture
and NaN for a covariance that is not positive definite."""
import ctypes as C
import os
import re
import shutil
import subprocess
import types
import warnings

import numpy as np
import pytest
from scipy.integrate import IntegrationWarning, quad
from scipy.special import ndtr

import corr_oracle as CO
import parity
from frenetix_occlusion_b200 import synthetic as S
from oracle import metric_oracle as MO

ARMED = {"harm": 0.1, "risk": 0.01, "be": 1.0, "cp": 0.05, "ttc": 2.0, "wttc": None, "ttce": None, "dce": 2.0}


# ---------------------------------------------------------------------------------------------------------------- CPU
def _quad_rect(a1, b1, a2, b2, r):
    s = np.sqrt(1.0 - r * r)
    f = lambda x: np.exp(-0.5 * x * x) / np.sqrt(2 * np.pi) * (ndtr((b2 - r * x) / s) - ndtr((a2 - r * x) / s))  # noqa: E731
    with warnings.catch_warnings():             # quad notes when roundoff stops it short of 1e-16; 1e-13 is checked
        warnings.simplefilter("ignore", IntegrationWarning)
        return quad(f, a1, b1, epsabs=1e-16, epsrel=1e-14, limit=200)[0]


def test_rectangle_mass_matches_quadrature_and_scipy():
    """The oracle's float64 rectangle mass (Genz's BVNU, the algorithm the kernels run) against the conditional form
    integrated by quad and against scipy's multivariate_normal.cdf (ref_shims.mvnun) over the whole rho range, with
    sigma_x != sigma_y and boxes at the mean and 1, 4 and 8 sigma away; at rho = 0 it is the diagonal closed form."""
    from oracle.ref_shims import mvnun
    sx, sy = 0.4, 1.3
    hx, hy = 0.75, 0.8                           # L/6, W/2 of the BMW 320i
    worst_q = worst_s = 0.0
    for r in (-0.99, -0.95, -0.8, -0.5, 0.0, 0.3, 0.6, 0.8, 0.93, 0.99):
        for dist in (0.0, 1.0, 4.0, 8.0):
            for ux, uy in ((1, 0), (0, 1), (1, 1), (-1, 1), (-1, -1)):
                cx, cy = ux * dist * sx, uy * dist * sy          # box centre relative to the mean
                a1, b1, a2, b2 = (cx - hx) / sx, (cx + hx) / sx, (cy - hy) / sy, (cy + hy) / sy
                got = float(CO.bvn_rect(a1, b1, a2, b2, r))
                worst_q = max(worst_q, abs(got - _quad_rect(a1, b1, a2, b2, r)))
                ref = mvnun([cx - hx, cy - hy], [cx + hx, cy + hy], [0.0, 0.0],
                            [[sx * sx, r * sx * sy], [r * sx * sy, sy * sy]])[0]
                worst_s = max(worst_s, abs(got - ref))
                if r == 0.0:
                    assert abs(got - (ndtr(b1) - ndtr(a1)) * (ndtr(b2) - ndtr(a2))) < 1e-15
    assert worst_q < 1e-13, worst_q
    assert worst_s < 1e-13, worst_s
    assert np.isnan(CO.bvn_rect(-1.0, 1.0, -1.0, 1.0, 1.0))


def _agent(cov, n=4):
    return {"agent_type": "Car", "length": 4.8, "width": 2.0, "buf_length": 5.76, "buf_width": 2.6,
            "pos": np.zeros((n, 2)), "yaw": np.zeros(n), "v": np.ones(n), "cov": np.asarray(cov, dtype=np.float64)}


def test_agent_set_validates_covariances():
    from frenetix_occlusion_b200.engine import AgentSet
    eye = np.array([[0.2, 0.0], [0.0, 0.5]])
    base = np.stack([eye] * 4)
    asym = base.copy()
    asym[2, 0, 1] = 0.1
    with pytest.raises(ValueError, match="symmetric"):
        AgentSet.from_case([_agent(asym)])
    for bad in (np.array([[0.2, 0.32], [0.32, 0.5]]),          # |rho| = 1.01
                np.array([[0.2, -0.32], [-0.32, 0.5]]),
                np.array([[0.2, np.sqrt(0.1)], [np.sqrt(0.1), 0.5]]),   # |rho| = 1
                np.array([[0.0, 0.1], [0.1, 0.5]]),            # zero variance with a covariance
                np.array([[0.0, 0.1], [0.1, 0.0]])):
        c = base.copy()
        c[1] = bad
        with pytest.raises(ValueError, match="positive definite"):
            AgentSet.from_case([_agent(c)])
    ok = base.copy()
    ok[1] = [[0.2, 0.3], [0.3, 0.5]]                           # rho = 0.95
    ok[3] = 0.0                                                # all zero: 0.1 I
    s = AgentSet.from_case([_agent(ok), _agent(base)])
    assert s.cov_xy is not None and s.cov_xy.shape == (2, 4)
    assert s.cov_xy[0, 1] == 0.3 and not s.cov_xy[1].any()
    # diagonal sets, with cov or with var, reach exactly what they reached before: no cov_xy, the same arrays
    d = AgentSet.from_case([_agent(base)])
    assert d.cov_xy is None
    v = _agent(base)
    del v["cov"]
    v["var"] = np.full(4, 0.3)
    d2 = AgentSet.from_case([v])
    assert d2.cov_xy is None and np.array_equal(d2.var_x, np.full((1, 4), 0.3))
    assert np.array_equal(d.var_x, [[0.2] * 4]) and np.array_equal(d.var_y, [[0.5] * 4])


def test_c_abi_argument_checks_without_device():
    from frenetix_occlusion_b200 import _lib as L
    for A, T in ((256, 51), (33, 31), (1, 1), (7, 3)):
        base = L.lib.fo_agent_table_bytes(A, T)
        assert L.lib.fo_agent_table_bytes_corr(A, T) == ((base + 15) & ~15) + A * T * 16
    assert L.lib.fo_agent_table_bytes_corr(-1, 4) == 0
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = 3, 5
    for f in ("x", "y", "yaw", "v", "var_x", "var_y", "n_states", "kind", "length", "width", "buf_length", "buf_width"):
        setattr(raw, f, p)
    veh = L.FoVehicle(4.5, 1.6, 1000.0, 1.4, 11.5)
    need = L.lib.fo_agent_table_bytes_corr(3, 5)
    assert L.lib.fo_agents_pack_corr(C.byref(raw), None, C.byref(veh), p, need, None) == -1      # NULL cov_xy
    assert b"NULL" in L.lib.fo_last_error()
    assert L.lib.fo_agents_pack_corr(C.byref(raw), p, C.byref(veh), None, need, None) == -1      # NULL table
    assert L.lib.fo_agents_pack_corr(C.byref(raw), p, C.byref(veh), p, need - 1, None) == -1     # too small
    assert L.lib.fo_agents_pack_corr(C.byref(raw), p, C.byref(veh), p, L.lib.fo_agent_table_bytes(3, 5), None) == -1
    assert b"too small" in L.lib.fo_last_error()
    assert L.lib.fo_metric_bundle_corr(None, None) == -1
    a = L.FoMetricArgs()
    a.n_traj, a.n_states, a.ego, a.valid, a.n_peers = 4, 31, p, p, 1
    assert L.lib.fo_metric_bundle_corr(C.byref(a), None) == -2                                   # peer stores
    a.n_peers, a.n_traj = 0, -1
    assert L.lib.fo_metric_bundle_corr(C.byref(a), None) == -1


def test_correlated_kernels_stay_inside_their_code_size_budgets():
    """The correlated kernels carry the float64 rectangle mass (bvn_rect and its out-of-line CDF / exp, about 18 kB)
    on top of the runtime-mask kernel they are built from.  Budgets: the sizes measured when they were added (DESIGN.md
    5.10) plus 4 kB."""
    from torch.utils.cpp_extension import CUDA_HOME
    from frenetix_occlusion_b200 import _lib as L
    cuobjdump = shutil.which("cuobjdump") or (CUDA_HOME and shutil.which("cuobjdump", path=os.path.join(CUDA_HOME, "bin")))
    if not cuobjdump:
        pytest.skip("cuobjdump not found (no CUDA toolkit)")
    sass = subprocess.run([cuobjdump, "-sass", L.LIB_PATH], capture_output=True, text=True).stdout
    sizes, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
        elif name and re.match(r"\s+/\*[0-9a-f]+\*/\s+\S", line):
            sizes[name] = sizes.get(name, 0) + 16

    def size_of(*parts):
        hit = [v for k, v in sizes.items() if all(p in k for p in parts)]
        assert len(hit) == 1, (parts, sorted(sizes))
        return hit[0]
    budget = {("fo_metric_sweep_corr_kernel", "ILb1ELb0E"): 71.375,   # one-warp window-filter shape
              ("fo_metric_sweep_corr_kernel", "ILb1ELb1E"): 83.75,  # ... with the float64 tie path
              ("fo_metric_sweep_corr_kernel", "ILb0ELb0E"): 82.0,  # team shape
              ("fo_metric_sweep_corr_kernel", "ILb0ELb1E"): 97.625,
              ("fo_metric_detail_corr_kernel",): 76.875}
    for parts, kb in budget.items():
        assert size_of(*parts) <= (kb + 4) * 1024, (parts, size_of(*parts))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _run(case, want_pair, want_step, agents=None):
    import torch
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]) if agents is None else agents)
    r = eng.assess(np.asarray(case["ego"]), want_pair=want_pair, want_step=want_step)
    torch.cuda.synchronize()
    res = {"valid": r.valid.cpu().numpy(), "summary": r.summary.cpu().numpy(), "flags": r.flags.cpu().numpy().astype(np.uint32)}
    res["pair"] = r.pair.cpu().numpy() if r.pair is not None else None
    res["step"] = r.step.cpu().numpy() if r.step is not None else None
    return res, eng


def _check(rep, max_tie_rate=0.005):
    assert not rep["fail"], "\n".join(rep["fail"])
    assert sum(rep["ties"].values()) <= max(3, max_tie_rate * rep["n_pairs"]), rep["ties"]


# (seed, N, A, T, metrics, thresholds, FO_TEAM_WARPS): A = 1 / 5 / 40 / 300, T = 2 / 31 / 51 / 128, both shapes (W = 1
# with >= 17 agents is the one-warp window-filter shape), default and all-7 metric sets, null and armed thresholds
CASES = [(1, 200, 1, 31, None, None, None), (2, 300, 5, 51, S.DEFAULT_METRICS, None, None),
         (3, 150, 40, 31, None, ARMED, "1"), (4, 60, 300, 51, None, None, "1"), (5, 100, 40, 128, None, None, None),
         (6, 80, 5, 2, None, ARMED, None), (7, 80, 300, 51, S.DEFAULT_METRICS, ARMED, "2"),
         (8, 120, 40, 51, S.DEFAULT_METRICS, None, "1"), (9, 20000, 5, 31, S.DEFAULT_METRICS, None, None)]


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,a,t,metrics,thr,warps", CASES)
def test_correlated_bundles_match_oracle(seed, n, a, t, metrics, thr, warps, cuda_device, monkeypatch):
    if warps:
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
    case = CO.add_correlations(S.make_case(n, a, t, seed=seed, activated_metrics=metrics, thresholds=thr), seed)
    out = CO.evaluate_bundle(case)
    res_s, eng = _run(case, False, False)
    assert eng._corr
    _check(parity.compare_bundle(out, res_s, case))                     # summary kernel: valid / summary / flags
    res_d, _ = _run(case, True, True)
    _check(parity.compare_bundle(out, res_d, case))                     # detail kernel: + pair / step
    assert np.isfinite(res_d["step"][..., 0]).all()


def _agent_manager(case):
    am = types.SimpleNamespace(dt=case["dt"], visualization=None, phantom_agents=[], predictions={})
    for k, ag in enumerate(case["agents"]):
        am.phantom_agents.append(types.SimpleNamespace(agent_id=10000 + k, agent_type=ag["agent_type"],
                                                       shape=types.SimpleNamespace(length=ag["length"], width=ag["width"])))
        am.predictions[int(str(10000 + k) + "0")] = {
            "orientation_list": np.asarray(ag["yaw"]), "v_list": np.asarray(ag["v"]),
            "pos_list": np.asarray(ag["pos"]).reshape(-1, 2), "shape": {"length": ag["buf_length"], "width": ag["buf_width"]},
            "cov_list": np.asarray(ag["cov"])}
    am.agent_by_prediction_id = lambda pid: next(x for x in am.phantom_agents if x.agent_id == int(str(pid)[:5]))
    return am


@pytest.mark.gpu
@pytest.mark.parametrize("prefetch", [False, True])
def test_metric_protocol_with_correlated_predictions(prefetch, cuda_device):
    """Metric.evaluate_metrics returns the reference's result dicts, per-step collision_probability arrays included,
    for predictions whose cov_list is correlated -- with and without Metric.prefetch; evaluate_bundle agrees."""
    from frenetix_occlusion_b200.metrics.metric import Metric
    from oracle.compare import compare_results
    from oracle.ref_runner import TrajectoryStub
    case = CO.add_correlations(S.make_case(40, 6, 31, seed=21), 21)
    for ag in case["agents"]:                                 # pull the agents onto the ego paths: many gated steps
        ag["pos"] = np.asarray(ag["pos"]) * 0.3
    out = CO.evaluate_bundle(case)
    metric = Metric({"activated_metrics": list(case["activated_metrics"]), "metric_thresholds": dict(case["thresholds"])},
                    types.SimpleNamespace(**case["vehicle"]), _agent_manager(case))
    trajs = [TrajectoryStub(case["ego"][n]) for n in range(40)]
    if prefetch:
        metric.prefetch(trajs)
    assert out["gate_fraction"] > 0.01
    for n, tr in enumerate(trajs):
        results, ok = metric.evaluate_metrics(tr)
        problems = compare_results(MO.to_reference_dict(out, n, case), results, rtol=1e-4, atol=2e-6)
        assert not problems, f"trajectory {n}:\n" + "\n".join(problems[:10])
        assert ok == bool(out["valid"][n])
    assert metric._core.engine._corr
    b = metric.evaluate_bundle(case["ego"])
    assert np.array_equal(b.valid.cpu().numpy().astype(bool), out["valid"])


@pytest.mark.gpu
def test_zero_correlation_table_matches_diagonal_path(cuda_device):
    """A correlated table with cov_xy = 0 packs the diagonal table byte for byte in front of its s3 section and gives
    the diagonal path's results within the parity tolerances (another CP function: not bit for bit)."""
    import torch
    from frenetix_occlusion_b200.engine import AgentSet
    case = S.make_case(300, 40, 31, seed=23)
    diag = AgentSet.from_case(case["agents"])
    zero = AgentSet.from_case(case["agents"])
    zero.cov_xy = np.zeros_like(zero.var_x)
    rd, ed = _run(case, True, True, diag)
    rz, ez = _run(case, True, True, zero)
    assert not ed._corr and ez._corr
    n = ed._table.numel()
    assert torch.equal(ez._table[:n], ed._table)
    assert np.array_equal(rz["valid"], rd["valid"]) and np.array_equal(rz["flags"], rd["flags"])
    np.testing.assert_allclose(rz["step"][..., 0], rd["step"][..., 0], rtol=parity.RTOL, atol=parity.ATOL_CP)
    np.testing.assert_allclose(rz["summary"], rd["summary"], rtol=parity.RTOL, atol=parity.ATOL_CP)
    rs, _ = _run(case, False, False, zero)
    rds, _ = _run(case, False, False, diag)
    np.testing.assert_allclose(rs["summary"], rds["summary"], rtol=parity.RTOL, atol=parity.ATOL_CP)
    assert np.array_equal(rs["valid"], rds["valid"])


@pytest.mark.gpu
@pytest.mark.parametrize("warps", [None, "1"])
def test_cuda_graph_replay_equals_eager(warps, cuda_device, monkeypatch):
    import torch
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    if warps:
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
    case = CO.add_correlations(S.make_case(1000, 32, 31, seed=25, thresholds=ARMED), 25)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    ego = eng.to_device_bundle(case["ego"]).clone()
    g, out = eng.capture(ego)
    eager = eng.assess(ego)
    torch.cuda.synchronize()
    ref = [x.clone() for x in (eager.valid, eager.summary.view(torch.int32), eager.flags)]
    for x in (out.valid, out.summary, out.flags):
        x.zero_()
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip((out.valid, out.summary.view(torch.int32), out.flags), ref):     # bits: NaN where BE overruns
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_not_positive_definite_gives_nan(cuda_device):
    """The C path does not inspect device data: a covariance with |rho| >= 1 gives NaN CP values, on the per-step
    detail and in max_collision_probability_all, instead of a plausible number."""
    from frenetix_occlusion_b200.engine import AgentSet
    case = S.make_case(200, 20, 31, seed=27, activated_metrics=["cp", "hr"])
    for ag in case["agents"]:
        ag["pos"] = np.asarray(ag["pos"]) * 0.3
    ag = AgentSet.from_case(case["agents"])
    ag.cov_xy = np.zeros_like(ag.var_x)
    ag.cov_xy[0] = 1.5 * np.sqrt(ag.var_x[0] * ag.var_y[0])      # agent 0: |rho| = 1.5 everywhere
    inside = MO.collision_probability(case)[1]
    assert inside[:, 0].any()
    rd, _ = _run(case, True, True, ag)
    cp = rd["step"][..., 0]
    assert np.isnan(cp[:, 0][inside[:, 0]]).all()
    assert np.isfinite(cp[:, 1:]).all()
    rs, _ = _run(case, False, False, ag)
    assert np.isnan(rs["summary"][inside[:, 0].any(1), 4]).all()


@pytest.mark.gpu
def test_batches_and_stats_refuse_correlated_sets(cuda_device):
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    case = CO.add_correlations(S.make_case(10, 4, 31, seed=29), 29)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    ag = AgentSet.from_case(case["agents"])
    with pytest.raises(ValueError, match="diagonal"):
        eng.set_agent_batch([ag, ag])
    eng.set_agents(ag)
    with pytest.raises(ValueError, match="diagonal"):
        eng.work_stats(case["ego"])
