"""Brake evaluation (BE) of the summary kernels as one walk over the pairs' common bisection tree (be_walk,
fo_metric_dev.cuh).

CPU: the float64 mirror of the walk in scripts/be_tree_count.py gives the same per-trajectory maximum and the same
range error as one bisection per pair with the running maximum as floor (the order the summary kernel used before).
GPU: on BE-heavy bundles the walk of the one-warp shape gives what one bisection per pair gives in the team shape, bit
for bit; its BE columns equal the maximum of the detail kernel's per-pair values; the results match the oracle; and the
batch entry point gives the same."""
import importlib.util
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from frenetix_occlusion_b200 import synthetic as S  # noqa: E402
from oracle import metric_oracle as MO  # noqa: E402


def _count_model():
    spec = importlib.util.spec_from_file_location("be_tree_count", os.path.join(ROOT, "scripts", "be_tree_count.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _ragged(case, seed):
    """Agents with fewer states than the ego, some with none at all."""
    rng = np.random.default_rng(seed)
    T = case["ego"].shape[1]
    for ag in case["agents"]:
        n = int(rng.choice([0, 1, max(1, T // 3), T - 1, T, T, T]))
        for k in ("pos", "yaw", "v", "var"):
            ag[k] = np.asarray(ag[k])[:n]
    return case


def _short_paths(case, every=3, scale=0.9):
    """Shrink every third planned path around its start: the re-timed paths then overrun (range errors)."""
    ego = case["ego"]
    sel = ego[::every]
    sel[..., 0:2] = sel[:, :1, 0:2] + scale * (sel[..., 0:2] - sel[:, :1, 0:2])
    ego[::every] = sel
    return case


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("seed,n,a,t,short", [(1, 150, 64, 51, False), (2, 150, 64, 51, True), (3, 120, 40, 31, True),
                                              (4, 60, 32, 128, False)])
def test_tree_walk_equals_per_pair_bisection(seed, n, a, t, short):
    M = _count_model()
    case = S.make_case(n, a, t, seed=seed)
    if short:
        _short_paths(case)
    stacked = MO._stack_agents(case)
    pairs = M.be_pairs(case)
    assert len(pairs) > n // 4
    n_err = 0
    for nidx, agents in pairs.items():
        tr = M.Trajectory(case, nidx, stacked)
        m0, e0, _ = M.per_pair(tr, agents)
        m1, e1, _ = M.tree_walk(tr, agents)
        assert e0 == e1, nidx
        if not e0:
            assert m0 == m1, (nidx, m0, m1)
        n_err += e0
    if short:
        assert n_err > 0


def test_tree_walk_tests_fewer_path_chunks():
    M = _count_model()
    case = S.make_case(80, 64, 51, seed=5)
    stacked = MO._stack_agents(case)
    pp = tw = 0
    for nidx, agents in M.be_pairs(case).items():
        tr = M.Trajectory(case, nidx, stacked)
        pp += M.per_pair(tr, agents)[2]["path_chunks"]
        tw += M.tree_walk(tr, agents)[2]["path_chunks"]
    assert 0 < tw < pp / 2, (tw, pp)


# ---------------------------------------------------------------------------------------------------- GPU
def _be_case(seed, n, a, t, armed):
    thr = dict(S.DEFAULT_THRESHOLDS)
    if armed:
        thr["be"] = 0.3
    case = S.make_case(n, a, t, seed=seed, thresholds=thr)
    _short_paths(case, every=5, scale=0.95)
    return _ragged(case, seed)


def _summary(case, monkeypatch, warps):
    import parity
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    return parity.run_gpu(case, want_pair=False, want_step=False)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("t", [2, 31, 51, 128])
@pytest.mark.parametrize("armed", [False, True])
def test_walk_equals_detail_maximum_and_team_split(t, armed, cuda_device, monkeypatch):
    import parity
    case = _be_case(100 + t, 400, 300, t, armed)           # 300 agents: three agent tiles
    res_d, _ = parity.run_gpu(case, want_pair=True, want_step=False)
    res_s = _summary(case, monkeypatch, 1)
    # the team shape bisects one pair at a time (be_bisect, pairs dealt round-robin to the warps): same maximum, same
    # range errors as the walk of the one-warp shape
    for warps in (2, 3, 8):
        res_w = _summary(case, monkeypatch, warps)
        for f in ("valid", "flags", "summary"):
            assert np.array_equal(res_w[f], res_s[f], equal_nan=f == "summary"), (warps, f)
    # against the per-pair bisections of the detail kernel, with the ties test_metric_gpu allows between the kernels
    same = res_d["flags"] == res_s["flags"]
    assert (~same).sum() <= max(2, 0.005 * len(same)), int((~same).sum())
    ok = ((res_d["flags"] & 1) == 0) & same
    assert np.array_equal(res_d["valid"][same], res_s["valid"][same])
    p = res_d["pair"]
    pmax = np.where(np.isnan(p[ok][..., 9]), 0.0, p[ok][..., 9]).max(1) if p.shape[1] else np.zeros(ok.sum())
    be_same = (pmax == res_s["summary"][ok, 9]) & (res_d["summary"][ok, 9] == res_s["summary"][ok, 9])
    assert (~be_same).sum() <= max(2, 0.005 * ok.sum()), int((~be_same).sum())
    # btn = max rcd / a_max, correctly rounded (the detail kernel's per-pair btn uses the approximate division)
    a_max = np.float32(case["vehicle"]["a_max"])
    assert np.array_equal(res_s["summary"][ok, 8], res_s["summary"][ok, 9] / a_max)
    assert np.all(np.isnan(res_s["summary"][(res_s["flags"] & 1) != 0, 8:10]))
    if t > 2:
        assert (res_s["summary"][ok, 9] > 0).sum() > 20          # the cases exercise BE


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,a,t,warps", [(201, 120, 300, 51, 1), (202, 150, 40, 31, 4), (203, 60, 33, 128, 1),
                                              (204, 200, 8, 2, 1)])
def test_walk_matches_oracle(seed, n, a, t, warps, cuda_device, monkeypatch):
    import parity
    from test_metric_gpu import _check
    case = _be_case(seed, n, a, t, armed=True)
    res = _summary(case, monkeypatch, warps)
    _check(parity.compare_bundle(MO.evaluate_bundle(case), res, case))


@pytest.mark.gpu
@pytest.mark.parametrize("warps", [1, 4])
def test_walk_through_the_batch_entry_point(warps, cuda_device, monkeypatch):
    import torch
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    cases = [_be_case(300 + i, n, a, 51, armed=bool(i & 1)) for i, (n, a) in enumerate([(300, 300), (50, 40), (1, 5)])]
    for c in cases[1:]:
        c["thresholds"] = cases[0]["thresholds"]
    eng = MetricEngine(cases[0]["vehicle"], 0.1, cases[0]["activated_metrics"], cases[0]["thresholds"])
    eng.set_agent_batch([AgentSet.from_case(c["agents"]) for c in cases])
    parts = eng.assess_batch([c["ego"] for c in cases]).split()
    single = MetricEngine(cases[0]["vehicle"], 0.1, cases[0]["activated_metrics"], cases[0]["thresholds"])
    for c, got in zip(cases, parts):
        single.set_agents(AgentSet.from_case(c["agents"]))
        want = single.assess(c["ego"])
        torch.cuda.synchronize()
        for f in ("valid", "flags", "summary"):
            g, w = getattr(got, f).cpu().numpy(), getattr(want, f).cpu().numpy()
            assert np.array_equal(g, w, equal_nan=f == "summary"), f
