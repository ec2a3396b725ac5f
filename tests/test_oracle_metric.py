"""Oracle B (vectorised float64 restatement) against the golden vectors produced by the
reference's own metric modules (oracle A, ``oracle/make_golden.py``), plus closed-form KATs
(SURVEY.md §8c).  CPU only."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_files
from oracle import metric_oracle as MO
from oracle.compare import compare_results
from oracle.geometry import ConvexPolygon, obb_distance, obb_intersects, rect_vertices


@pytest.mark.parametrize("fname", golden_files("metric_"))
def test_oracle_b_matches_reference_golden(fname):
    case, reference, order = MO.load_case_json(os.path.join(GOLDEN, fname))
    out = MO.evaluate_bundle(case)
    assert out["order"] == order
    for n, ref in enumerate(reference):
        if ref["safety_check"] is None:           # the reference raised (BE interp1d bounds)
            assert out["be_error"][n], f"{fname}[{n}]: reference raised but oracle B did not flag it"
            continue
        assert not out["be_error"][n]
        got = MO.to_reference_dict(out, n, case)
        problems = compare_results(ref["results"], got, rtol=1e-12, atol=1e-15)
        assert not problems, f"{fname}[{n}]:\n" + "\n".join(problems[:10])
        assert bool(out["valid"][n]) == ref["safety_check"], f"{fname}[{n}] safety_check"


def test_kat_values_from_survey():
    case, reference, _ = MO.load_case_json(os.path.join(GOLDEN, "metric_kat_pedestrian.json"))
    out = MO.evaluate_bundle(case)
    assert out["dce"][0, 0] == 0.0 and out["time_dce"][0, 0] == 15
    assert out["ttc"][0, 0] == 1.5 and out["ttce"][0, 0] == 1.5 and out["wttc"][0] == 1.5
    assert out["be_rcd"][0, 0] == 4.609375
    assert abs(out["max_collision_probability_all"][0] - 0.4925777927) < 1e-6
    assert abs(out["max_obst_harm_with_cp_all"][0] - 0.2738569749) < 1e-6
    assert not out["valid"][0]                    # harm 0.1 threshold -> rejected (README.md:19-25)


def test_closed_form_geometry():
    # axis-aligned gap g -> round(g, 3); overlap -> 0; containment -> 0
    d = obb_distance(0.0, 0.0, 0.0, 2.0, 1.0, 5.25, 0.0, 0.0, 1.0, 1.0)
    assert abs(float(d) - 2.25) < 1e-15
    assert float(obb_distance(0.0, 0.0, 0.0, 2.0, 1.0, 0.2, 0.1, 0.7, 0.3, 0.2)) == 0.0
    assert bool(obb_intersects(0.0, 0.0, 0.0, 2.0, 1.0, 3.0, 0.0, 0.0, 1.0, 1.0))   # touching counts
    assert not bool(obb_intersects(0.0, 0.0, 0.0, 2.0, 1.0, 3.0 + 1e-9, 0.0, 0.0, 1.0, 1.0))


def test_two_geometry_formulations_agree():
    rng = np.random.default_rng(5)
    for _ in range(300):
        ax, ay, bx, by = rng.uniform(-6, 6, 4)
        aw, bw = rng.uniform(-np.pi, np.pi, 2)
        al, awd, bl, bwd = rng.uniform(0.3, 5.0, 4)
        pa = ConvexPolygon(rect_vertices(ax, ay, al, awd, aw))
        pb = ConvexPolygon(rect_vertices(bx, by, bl, bwd, bw))
        d_box = float(obb_distance(ax, ay, aw, al / 2, awd / 2, bx, by, bw, bl / 2, bwd / 2))
        assert abs(pa.distance(pb) - d_box) < 1e-12
        assert pa.intersects(pb) == bool(obb_intersects(ax, ay, aw, al / 2, awd / 2, bx, by, bw, bl / 2, bwd / 2))


def test_mass_and_lr4s_boundaries():
    assert abs(MO.obstacle_mass("car", 4.8 * 1.2 * 2.0 * 1.3) - (-1333.5 + 526.9 * 14.976 ** 0.8)) < 1e-9
    assert MO.obstacle_mass("pedestrian", 1.0) == 75 and MO.obstacle_mass("bicycle", 1.0) == 90
    assert MO.check_required_metrics(["hr", "ttc", "ttce", "dce", "wttc", "cp"]) == \
        ["cp", "dce", "ttc", "hr", "ttce", "wttc"]
    assert MO.check_required_metrics(["hr", "ttc", "be", "ttce", "dce", "wttc", "cp"]) == \
        ["cp", "dce", "ttc", "hr", "be", "ttce", "wttc"]


def test_no_agents_is_valid():
    case, _, _ = MO.load_case_json(os.path.join(GOLDEN, "metric_kat_pedestrian.json"))
    case["agents"] = []
    out = MO.evaluate_bundle(case)
    assert out["valid"].all()                     # metric.py:44-45


def test_varied_agents_reach_what_agent_table_does_not():
    """Every kind of the C ABI, headings outside [-pi, pi], changing heading and speed, var_x != var_y, all-zero
    covariances and ragged lengths, all float32-representable; a parked vehicle does not move."""
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200 import synthetic as S
    for jitter in (False, True):
        ags = S.varied_agents(60, 31, 3, jitter=jitter)
        assert {a["agent_type"].lower() for a in ags} == set(L.KINDS)
        assert {len(a["yaw"]) for a in ags} == {1, 2, 8, 9, 31, 51}
        assert any((np.abs(a["yaw"]) > np.pi).any() for a in ags)
        moving = [a for a in ags if len(a["yaw"]) > 2 and a["agent_type"] != "ParkedVehicle"]
        assert all(np.ptp(a["yaw"]) > 0 and np.ptp(a["v"]) > 0 for a in moving)
        assert all(not a["v"].any() for a in ags if a["agent_type"] == "ParkedVehicle")
        cov = np.concatenate([a["cov"] for a in ags])
        assert not cov[:, [0, 1], [1, 0]].any() and (cov[:, 0, 0] != cov[:, 1, 1]).mean() > 0.8
        zero = (cov == 0).all((1, 2))
        assert 0.05 < zero.mean() < 0.15 and ((cov[:, 0, 0] == 0) == zero).all() and ((cov[:, 1, 1] == 0) == zero).all()
        for a in ags:
            for k in ("pos", "yaw", "v", "var", "cov"):
                assert np.array_equal(S._f32(a[k]), a[k])
            assert np.array_equal(a["var"], a["cov"][:, 0, 0])
            if a["agent_type"] in ("Car", "PriorityVehicle", "ParkedVehicle", "Taxi"):
                assert MO.obstacle_mass(a["agent_type"], a["buf_length"] * a["buf_width"]) > 0


def test_oracle_b_per_axis_covariance():
    """Oracle B's collision probability with a diagonal ``cov`` (sigma_x = sqrt(cov[i-1][0][0]), sigma_y =
    sqrt(cov[i-1][1][1])) equals the correlated oracle at rho = 0 (pinned to scipy and quadrature in test_metric_corr)
    on every step, and the reference's nine mvnun terms (``ref_shims.mvnun``) on gated steps with var_x != var_y.
    A correlated covariance is refused."""
    import corr_oracle as CO
    from frenetix_occlusion_b200 import synthetic as S
    from oracle.ref_shims import mvnun
    for jitter in (False, True):
        case = S.make_varied_case(300, 40, 31, seed=11 + jitter, jitter=jitter)
        cp, inside, _ = MO.collision_probability(case)
        cp_c, inside_c, _ = CO.collision_probability(case)
        assert np.array_equal(inside, inside_c) and inside.mean() > 0.01
        assert np.abs(cp - cp_c).max() <= 1e-13
        ego, L, W = case["ego"], case["vehicle"]["length"], case["vehicle"]["width"]
        rng = np.random.default_rng(3)
        hits = np.argwhere(inside & (cp > 1e-3))
        checked = 0
        for n, a, j in hits[rng.permutation(len(hits))]:
            ag, i = case["agents"][a], j + 1
            c = ag["cov"][i - 1]
            if c[0, 0] == c[1, 1] or c[0, 0] == 0:
                continue
            h = np.array([np.cos(ag["yaw"][i]), np.sin(ag["yaw"][i])]) * ag["buf_length"] / 2
            p = ag["pos"][i - 1]
            e, th = ego[n, i, :2], ego[n, i, 2]
            off = np.array([np.cos(th), np.sin(th)]) * L / 3
            half = np.array([L / 6, W / 2])
            want = sum(mvnun(b - half, b + half, mu, c)[0] for mu in (p, p + h, p - h) for b in (e, e + off, e - off)) / 3
            assert abs(cp[n, a, j] - want) <= 1e-13 * max(1.0, want), (n, a, j)
            checked += 1
            if checked == 12:
                break
        assert checked == 12
    case["agents"][3]["cov"] = case["agents"][3]["cov"].copy()
    case["agents"][3]["cov"][5, 0, 1] = case["agents"][3]["cov"][5, 1, 0] = 0.01
    with pytest.raises(ValueError, match="correlated"):
        MO.collision_probability(case)
