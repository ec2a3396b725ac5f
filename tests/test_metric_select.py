"""The first valid row of each problem of a batch (fo_metric_batch_select, MetricEngine.select_batch / select,
Metric.select, FOInterface.select_trajectory, batch.select_interfaces).

CPU: declaration and export, every argument check without a device, code-size budgets of the new kernels.  GPU (-m gpu):
selected equals the first valid row of fo_metric_batch[_corr] on the same arguments; rows up to it are bit-identical
to that call's, later rows are identical or FO_VALID_SKIPPED; controlled first-valid positions; a large bundle assesses
far fewer rows than it has; on the golden scene fans the interface calls equal the first valid row of assess_bundle."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from kernel_sizes import size_of
from test_metric_batch import _batch_args
from test_metric_batch_corr import _flags, _mixed, _vehicles
from test_metric_batch_vehicles import _malformed_summary_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2
ARMED = {"harm": 0.1, "risk": 0.01, "be": 1.0, "cp": 0.05, "ttc": 2.0, "wttc": None, "ttce": None, "dce": 2.0}


# ---------------------------------------------------------------------------------------------------- CPU
def test_select_is_declared_and_exported():
    from frenetix_occlusion_b200 import _lib as L
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fo_b200.h")).read(), flags=re.S)
    assert re.search(r"\bfo_metric_batch_select\s*\(", text)
    assert re.search(r"#define\s+FO_VALID_SKIPPED\s+2\b", text) and L.FO_VALID_SKIPPED == 2
    assert "fo_metric_batch_select" in L.EXPORTED_SYMBOLS and hasattr(L.lib, "fo_metric_batch_select")


def test_select_checks_its_arguments_without_device():
    from frenetix_occlusion_b200 import _lib as L
    f = L.lib.fo_metric_batch_select
    sel = (C.c_int32 * 16)()
    sel_p = C.cast(sel, C.c_void_p)
    fleet = _vehicles(L, 8)
    # the malformed descriptors of fo_metric_batch_vehicles, with and without flags / vehicles: the same status
    for name, a in _malformed_summary_cases(L):
        old = L.lib.fo_metric_batch_vehicles(C.byref(a), fleet, None)
        for flags in (None, _flags(8, 0), _flags(8, 1)):
            for veh in (None, fleet):
                assert old != 0 and f(C.byref(a), flags, veh, sel_p, None) == old, name
                assert b"fo_metric_batch_select" in L.lib.fo_last_error()
    assert f(None, None, None, sel_p, None) == FO_ERR_INVALID_ARG
    # selected_dev: NULL or misaligned with problems
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    assert f(C.byref(a), None, None, None, None) == FO_ERR_INVALID_ARG
    assert b"selected_dev" in L.lib.fo_last_error()
    assert f(C.byref(a), None, None, C.c_void_p(sel_p.value + 2), None) == FO_ERR_INVALID_ARG
    # pair / step / peers: unsupported, before the selected_dev check and any device work
    for field, value in (("pair", 1 << 24), ("step", 1 << 24), ("n_peers", 1)):
        a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
        setattr(a.common, field, value)
        assert f(C.byref(a), None, None, sel_p, None) == FO_ERR_UNSUPPORTED, field
        assert f(C.byref(a), None, None, None, None) == FO_ERR_UNSUPPORTED, field
    # a flagged table is checked against the correlated size
    A, T = 5, 31
    arena_bytes = (L.lib.fo_agent_table_bytes(A, T) + 15) // 16 * 16
    a = _batch_args(L, [(0, 4, A, T, 0)], 4, arena_bytes=arena_bytes)
    assert f(C.byref(a), _flags(1, 1), None, sel_p, None) == FO_ERR_INVALID_ARG
    assert b"correlated table of problem 0" in L.lib.fo_last_error()
    # no problems: nothing is read
    e = _batch_args(L, [], 0)
    assert f(C.byref(e), None, None, None, None) == 0


def test_select_kernels_stay_inside_their_code_size_budgets():
    """fo_metric_batch_select_kernel is fo_metric_batch_kernel<0> / fo_metric_batch_corr_kernel plus the rank-major
    claim map and three early-exit checks.  Budgets: the sizes measured when they were added (DESIGN.md 5.14) + 4 kB."""
    budget = {"ILb1ELb0ELb0E": 54.0, "ILb1ELb1ELb0E": 67.875, "ILb0ELb0ELb0E": 63.375, "ILb0ELb1ELb0E": 79.625,
              "ILb1ELb0ELb1E": 76.5, "ILb1ELb1ELb1E": 88.875, "ILb0ELb0ELb1E": 86.125, "ILb0ELb1ELb1E": 101.375}
    for tmpl, kb in budget.items():
        size = size_of("fo_metric_batch_select_kernel", tmpl)
        assert size <= (kb + 4) * 1024, (tmpl, size)


# ---------------------------------------------------------------------------------------------------- GPU
def _host(r):
    return r.valid.cpu().numpy(), r.summary.view(__import__("torch").int32).cpu().numpy(), r.flags.cpu().numpy()


def _filled(eng_out_like):
    """Outputs of the batch's size prefilled with marker values (so an unwritten valid byte shows)."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import BatchResult
    N, dev = int(eng_out_like.valid.numel()), eng_out_like.valid.device
    return BatchResult(torch.full((N,), 7, dtype=torch.uint8, device=dev),
                       torch.full((N, L.FO_SUMMARY_K), -3.0, dtype=torch.float32, device=dev),
                       torch.full((N,), -5, dtype=torch.int32, device=dev), eng_out_like.offsets)


def _assert_select_matches(full, got):
    """got (select) against full (the batch call on the same arguments): selected, bits up to it, skips after it."""
    fv, fs, ff = _host(full)
    gv, gs, gf = _host(got)
    sel = got.selected.cpu().numpy()
    off = [int(x) for x in full.offsets]
    assert len(sel) == len(off) - 1
    n_assessed = 0
    for p in range(len(off) - 1):
        lo, hi = off[p], off[p + 1]
        ok = np.flatnonzero(fv[lo:hi] == 1)
        want = int(ok[0]) if len(ok) else hi - lo
        assert sel[p] == want, (p, sel[p], want, hi - lo)
        head = slice(lo, lo + min(want + 1, hi - lo))
        assert np.array_equal(gv[head], fv[head]) and np.array_equal(gs[head], fs[head]) and \
            np.array_equal(gf[head], ff[head]), p
        tail = np.arange(lo + want + 1, hi)
        skipped = gv[tail] == 2
        same = (gv[tail] == fv[tail]) & (gs[tail] == fs[tail]).all(axis=1) & (gf[tail] == ff[tail])
        assert np.all(skipped | same), p
        n_assessed += int((gv[lo:hi] != 2).sum())
    assert set(np.unique(gv)) <= {0, 1, 2}
    return n_assessed


def _batch_engine_for(probs, fleet):
    from test_metric_batch_corr import _engine
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet, correlated=True)
    return eng


def _run(eng, egos):
    import torch
    full = eng.assess_batch(egos)
    full.valid, full.summary, full.flags = full.valid.clone(), full.summary.clone(), full.flags.clone()
    got = eng.select_batch(egos, out=_filled(full))
    torch.cuda.synchronize()
    return full, got


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("warps", [1, 4])
@pytest.mark.parametrize("every", [0, 1, 2], ids=["diagonal", "correlated", "mixed"])
def test_selected_is_the_first_valid_row_of_the_batch_call(T, warps, every, cuda_device, monkeypatch):
    """Problems with 0, 1, 17 and 40 agents and 0, 1, 31 and 1000 rows, one vehicle each, armed thresholds (so rows
    fail), in batches of 1, 3 and 17 problems."""
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    for P in (1, 3, 17):
        probs, fleet = _mixed(T * 7 + P + every, T, a_set=(0, 1, 17, 40), n_set=(0, 1, 31, 1000), n_problems=P,
                              thresholds=ARMED, every=every)
        eng = _batch_engine_for(probs, fleet)
        full, got = _run(eng, [p[2] for p in probs])
        _assert_select_matches(full, got)


@pytest.mark.gpu
@pytest.mark.parametrize("warps", [1, 4])
@pytest.mark.parametrize("every", [0, 1, 2], ids=["diagonal", "correlated", "mixed"])
def test_selected_is_the_first_valid_row_of_the_batch_call_on_varied_agents(warps, every, cuda_device, monkeypatch):
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    for P in (1, 3, 17):
        probs, fleet = _mixed(P + every + 900, 51, a_set=(0, 1, 17, 40), n_set=(0, 1, 31, 1000), n_problems=P,
                              thresholds=ARMED, every=every, varied=True)
        full, got = _run(_batch_engine_for(probs, fleet), [p[2] for p in probs])
        _assert_select_matches(full, got)


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", [None, "default"], ids=["all", "default"])
@pytest.mark.parametrize("armed", [False, True], ids=["null", "armed"])
def test_selected_with_metric_sets_and_thresholds(metrics, armed, cuda_device, monkeypatch):
    from frenetix_occlusion_b200 import synthetic as S
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    probs, fleet = _mixed(71 + armed, 31, a_set=(1, 17, 40, 0), n_set=(31, 1000, 1), n_problems=9,
                          metrics=S.DEFAULT_METRICS if metrics else None, thresholds=ARMED if armed else None)
    eng = _batch_engine_for(probs, fleet)
    full, got = _run(eng, [p[2] for p in probs])
    _assert_select_matches(full, got)


@pytest.mark.gpu
def test_selected_with_a_covariance_that_is_not_positive_definite(cuda_device, monkeypatch):
    """NaN collision probabilities in one problem's rows: the select call follows the batch call's valid bytes."""
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    probs, fleet = _mixed(89, 31, a_set=(20, 5, 40, 3), n_set=(120, 64), n_problems=6, metrics=["cp", "hr"],
                          thresholds=ARMED)
    case = S.make_case(120, 20, 31, seed=89, activated_metrics=["cp", "hr"], thresholds=ARMED)
    for a in case["agents"]:
        a["pos"] = np.asarray(a["pos"]) * 0.3
    ag = AgentSet.from_case(case["agents"])
    ag.cov_xy = np.zeros_like(ag.var_x)
    ag.cov_xy[0] = 1.5 * np.sqrt(ag.var_x[0] * ag.var_y[0])
    probs[2] = (ag, (0.0, 0.0), case["ego"], case)
    eng = _batch_engine_for(probs, fleet)
    full, got = _run(eng, [p[2] for p in probs])
    assert np.isnan(full.summary.cpu().numpy()[int(full.offsets[2]):int(full.offsets[3]), 4]).any()
    _assert_select_matches(full, got)


def _reordered_case(n, a, t, seed, corr):
    """A case with armed thresholds and its rows' valid bytes from one full pass (engine on its own table)."""
    import corr_oracle as CO
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    case = S.make_case(n, a, t, seed=seed, thresholds={**ARMED, "harm": 0.1})
    if corr:
        case = CO.add_correlations(case, seed)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    valid = eng.assess(case["ego"]).valid.cpu().numpy()
    return eng, case["ego"], valid


@pytest.mark.gpu
@pytest.mark.parametrize("corr", [False, True], ids=["diagonal", "correlated"])
def test_controlled_first_valid_positions(corr, cuda_device):
    """Rows reordered so the first valid one is at rank 0, N/2 and N-1; with no valid row every output is the full
    call's."""
    import torch
    eng, ego, valid = _reordered_case(1000, 24, 31, 5 + corr, corr)
    good, bad = np.flatnonzero(valid == 1), np.flatnonzero(valid == 0)
    assert len(good) >= 1 and len(bad) >= 10, (len(good), len(bad))
    N = len(bad) + 1
    for pos in (0, N // 2, N - 1):
        order = np.concatenate([bad[:pos], good[:1], bad[pos:]])
        e = ego[order]
        full = eng.assess(e)
        r = eng.select(e)
        torch.cuda.synchronize()
        full.offsets = r.offsets
        assert int(r.selected.item()) == pos
        _assert_select_matches(full, r)
    e = ego[bad]
    full = eng.assess(e)
    r = eng.select(e)
    torch.cuda.synchronize()
    assert int(r.selected.item()) == len(bad)
    for g, w in zip(_host(r), _host(full)):
        assert np.array_equal(g, w)


@pytest.mark.gpu
def test_a_large_bundle_assesses_few_rows_when_an_early_row_is_valid(cuda_device):
    import torch
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    N = 200_000
    case = S.make_case(N, 64, 31, seed=17)
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
    eng.set_agents(AgentSet.from_case(case["agents"]))
    head = eng.assess(case["ego"][:64]).valid.cpu().numpy()
    assert head.any()
    r = eng.select(case["ego"])
    torch.cuda.synchronize()
    k = int(r.selected.item())
    assert k == int(np.flatnonzero(head)[0])
    assessed = int((r.valid != 2).sum().item())
    assert assessed < N // 4, assessed


# ---- interfaces ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_select_trajectory_equals_the_first_valid_candidate_on_the_scene_fans(cuda_device):
    from test_metric_batch_corr import _corr_scenes
    from test_metric_batch_detail import _trajectories
    fos, fans = _corr_scenes()
    for i, (fo, fan) in enumerate(zip(fos, fans)):
        cands = _trajectories(fan)
        valid = fo.assess_bundle(fan).valid.cpu().numpy()
        first = int(np.flatnonzero(valid)[0]) if valid.any() else None
        loop = next((k for k, t in enumerate(cands) if fo.trajectory_safety_assessment(t)[1]), None)
        assert loop == first, (i, loop, first)           # no documented summary / detail tie on these fans
        assert fo.select_trajectory(fan) == first, i
        assert fo.select_trajectory(cands) == first, i
        # the same candidates from the first valid one on, and a list with none valid
        if first is not None:
            assert fo.select_trajectory(fan[first:]) == 0
            bad = [t for t, v in zip(cands, valid) if not v]
            if bad:
                assert fo.select_trajectory(bad) is None
        assert fo.select_trajectory([]) is None


@pytest.mark.gpu
def test_select_interfaces_equals_each_interface(cuda_device):
    from frenetix_occlusion_b200.batch import select_interfaces
    from test_metric_batch_corr import _corr_scenes
    fos, fans = _corr_scenes()
    want = [fo.select_trajectory(f) for fo, f in zip(fos, fans)]
    assert select_interfaces(fos, fans) == want
    rev = [f[::-1].copy() for f in fans]
    assert select_interfaces(fos, rev) == [fo.select_trajectory(f) for fo, f in zip(fos, rev)]
