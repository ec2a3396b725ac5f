"""Parity of the dense metric core on agent predictions that turn, change speed, carry per-axis variances and cover
every obstacle type (``synthetic.varied_agents``), against the float64 oracles.  Needs a GPU.

The phantom agents of ``synthetic.agent_table`` and the reference's golden fixtures keep heading and speed constant,
use one variance for both axes and are Pedestrian, Bicycle, Car or Truck.  On such inputs a kernel that takes a
heading or speed from the neighbouring step, swaps sigma_x and sigma_y, or misreads the mass or protection of Bus,
Motorcycle, Train, PriorityVehicle, ParkedVehicle, Taxi or Unknown gives the right answer.  Here each of those
mistakes changes the result.

What the kernels are compared with here is oracle B's reading of the reference, not the reference itself: the step
from which the collision probability takes the agent's heading (state i) and position and covariance (state i-1),
collision_probability.py:51-52, and the step of the heading, speed and position in the harm, harm_model.py:81-97.
The golden fixtures never exercised those index conventions, because their headings and speeds are constant; no
fixture from the reference's own run covers these inputs yet.
"""
import types

import numpy as np
import pytest

import corr_oracle as CO
import parity
from frenetix_occlusion_b200 import synthetic as S
from oracle import metric_oracle as MO
from test_metric_gpu import _check, assert_summary_equals_detail

pytestmark = pytest.mark.gpu


def varied_case(n, a, t, seed, jitter=False, metrics=None, thresholds=None, **kw):
    return S.make_varied_case(n, a, t, seed=seed, activated_metrics=metrics, thresholds=thresholds, jitter=jitter, **kw)


def _summary_vs_oracle(case):
    out = MO.evaluate_bundle(case)
    res, eng = parity.run_gpu(case, want_pair=False, want_step=False)
    assert eng.agents.cov_xy is None and not eng._corr          # the diagonal kernels
    _check(parity.compare_bundle(out, res, case))
    return out


@pytest.mark.parametrize("seed,n,a,t", [(101, 300, 40, 2), (102, 300, 5, 9), (103, 100, 300, 31), (104, 200, 40, 51),
                                        (105, 200, 1, 128), (106, 300, 1, 31), (107, 100, 40, 128), (108, 100, 300, 9),
                                        (109, 300, 5, 51)])
@pytest.mark.parametrize("jitter", [False, True], ids=["kinematic", "jitter"])
def test_summary_kernel_team_shape(seed, n, a, t, jitter, cuda_device):
    """The default (multi-warp team) shape at 1 / 5 / 40 / 300 agents (more than one 256-agent tile) and T from 2 to
    FO_MAX_STATES."""
    out = _summary_vs_oracle(varied_case(n, a, t, seed, jitter))
    if t > 2 and a > 1:
        assert out["gate_fraction"] > 0.005 and out["max_collision_probability_all"].max() > 0.05


@pytest.mark.parametrize("metrics", [None, S.DEFAULT_METRICS, ["hr", "cp"]], ids=["all", "default", "hr-cp"])
@pytest.mark.parametrize("jitter", [False, True], ids=["kinematic", "jitter"])
def test_window_filter_shape(metrics, jitter, cuda_device, monkeypatch):
    """One warp per trajectory with >= 17 agents: the (agent, 8-step window) filter bounds speeds by the window's
    largest |v|, which only changing speeds put to the test."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    _summary_vs_oracle(varied_case(300, 40, 51, 111 + jitter, jitter, metrics))


@pytest.mark.parametrize("jitter", [False, True], ids=["kinematic", "jitter"])
def test_armed_distance_thresholds_on_the_window_filter_shape(jitter, cuda_device, monkeypatch):
    """The float64 tie variant of the one-warp shape: with dce / ttc armed the mask equals the oracle's bit for bit."""
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    thresholds = {"harm": None, "risk": None, "be": None, "cp": None, "wttc": None, "ttce": None, "dce": 0.75, "ttc": 1.2}
    # every trajectory starts at the origin: agents kept 8 m ahead of it leave some trajectories valid
    case = varied_case(1500, 40, 51, 121 + jitter, jitter, thresholds=thresholds, area=((8.0, 60.0), (-30.0, 30.0)))
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=False, want_step=False)
    rep = parity.compare_bundle(out, res, case)
    assert not rep["fail"], "\n".join(rep["fail"])
    ok = ~out["be_error"] & ((res["flags"] & 1) == 0)
    assert np.array_equal(res["valid"].astype(bool)[ok], out["valid"][ok])
    assert np.array_equal(np.round(res["summary"][ok, 6].astype(np.float64), 3), out["dce"].min(1)[ok])
    assert 0 < out["valid"].sum() < len(out["valid"])


@pytest.mark.parametrize("seed,n,a,t", [(131, 300, 40, 31), (132, 200, 23, 51), (133, 200, 11, 9)])
@pytest.mark.parametrize("jitter", [False, True], ids=["kinematic", "jitter"])
def test_detail_kernel(seed, n, a, t, jitter, cuda_device):
    """Per-step CP, ego and obstacle harm, the per-pair maxima, the risk argmax and BE of the detail kernel."""
    case = varied_case(n, a, t, seed, jitter)
    out = MO.evaluate_bundle(case)
    res, _ = parity.run_gpu(case, want_pair=True, want_step=True)
    rep = parity.compare_bundle(out, res, case)
    _check(rep)
    assert rep["n_be_pairs"] > 0 and np.isfinite(res["step"][..., :3][~np.isnan(out["ego_harm"])]).all()


@pytest.mark.parametrize("jitter", [False, True], ids=["kinematic", "jitter"])
def test_summary_kernel_equals_detail_kernel(jitter, cuda_device):
    """At a size the oracle would need minutes for."""
    assert_summary_equals_detail(varied_case(3000, 300, 51, 141 + jitter, jitter))


@pytest.mark.parametrize("seed,n,a,t,warps", [(151, 200, 40, 31, None), (152, 150, 40, 51, "1"), (153, 200, 5, 9, None)])
def test_correlated_kernels(seed, n, a, t, warps, cuda_device, monkeypatch):
    """The correlated (float64 CP) kernel family, summary and detail, on varied agents given correlations."""
    if warps:
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
    case = CO.add_correlations(varied_case(n, a, t, seed, jitter=seed % 2 == 0), seed)
    out = CO.evaluate_bundle(case)
    for detail in (False, True):
        res, eng = parity.run_gpu(case, want_pair=detail, want_step=detail)
        assert eng._corr
        _check(parity.compare_bundle(out, res, case))


@pytest.mark.parametrize("jitter", [False, True], ids=["kinematic", "jitter"])
def test_metric_protocol(jitter, cuda_device):
    """``Metric.evaluate_metrics`` on predictions with varying orientation_list / v_list and a diagonal cov_list with
    unequal axes returns the reference's result dicts; the set stays on the diagonal path."""
    from frenetix_occlusion_b200.metrics.metric import Metric
    from oracle.compare import compare_results
    from oracle.ref_runner import TrajectoryStub
    from test_metric_corr import _agent_manager
    case = varied_case(40, 12, 31, 161 + jitter, jitter)
    for ag in case["agents"]:                     # pull the agents onto the ego paths: many gated steps
        ag["pos"] = S._f32(np.asarray(ag["pos"]) * 0.3)
    out = MO.evaluate_bundle(case)
    assert out["gate_fraction"] > 0.01
    metric = Metric({"activated_metrics": list(case["activated_metrics"]), "metric_thresholds": dict(case["thresholds"])},
                    types.SimpleNamespace(**case["vehicle"]), _agent_manager(case))
    pids = list(metric.agent_manager.predictions)
    n_ties = 0
    for n in range(len(case["ego"])):
        if out["be_error"][n]:                    # the reference raises from interp1d (be.py:116-124)
            with pytest.raises(ValueError):
                metric.evaluate_metrics(TrajectoryStub(case["ego"][n]))
            continue
        results, ok = metric.evaluate_metrics(TrajectoryStub(case["ego"][n]))
        ref = MO.to_reference_dict(out, n, case)
        hr = results["hr"]
        gi = np.array([hr[p]["max_obst_risk_index"] if p in hr else 0 for p in pids])
        for k in np.nonzero(parity.risk_index_tie({"obst_risk": out["obst_risk"][n]}, gi))[0]:
            if pids[k] in hr and hr[pids[k]]["max_obst_risk_index"] != ref["hr"][pids[k]]["max_obst_risk_index"]:
                hr[pids[k]]["max_obst_risk_index"] = ref["hr"][pids[k]]["max_obst_risk_index"]     # a counted tie
                n_ties += 1
        problems = compare_results(ref, results, rtol=1e-4, atol=2e-6)
        assert not problems, f"trajectory {n}:\n" + "\n".join(problems[:10])
        assert ok == bool(out["valid"][n])
    assert n_ties <= 3
    eng = metric._core.engine
    assert eng.agents.cov_xy is None and not eng._corr and (eng.agents.var_x != eng.agents.var_y).any()
