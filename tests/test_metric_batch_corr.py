"""Correlated and diagonal prediction covariances in one batch of independent planning problems
(fo_agent_batch_layout_corr, fo_agents_pack_batch_corr, fo_metric_batch_corr, fo_metric_batch_detail_corr,
MetricEngine.set_agent_batch(correlated=True), and batch.assess_interfaces / prefetch_interfaces over interfaces whose
predictions carry correlated covariances).  The CPU part checks the layout, the argument validation (before any CUDA
call) and the code size of the new kernels; the GPU part checks that every problem of a mixed batch gets exactly what
the single-problem path gives it: fo_agents_pack_corr + fo_metric_bundle_corr when correlated, fo_agents_pack +
fo_metric_bundle when not."""
import copy
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import corr_oracle as CO
import parity
from test_metric_batch import _batch_args, _problems
from test_metric_batch_detail import SCENES, _assert_same_assessments, _trajectories
from test_metric_batch_vehicles import (_assert_equal, _engine, _fleet, _malformed_detail_cases, _malformed_summary_cases,
                                        _scene_interface_with)

FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2


def _flags(n, value):
    return (C.c_uint8 * max(n, 1))(*([value] * n))


def _vehicles(L, n):
    return (L.FoVehicle * max(n, 1))(*[L.FoVehicle(4.5, 1.6, 1200.0, 1.4, 10.0) for _ in range(n)])


# ---------------------------------------------------------------------------------------------------- CPU
def test_layout_of_correlated_tables():
    from frenetix_occlusion_b200 import _lib as L
    n_agents = np.array([3, 0, 40, 1, 300, 7], dtype=np.int32)
    t_stride = np.array([31, 31, 51, 2, 128, 0], dtype=np.int32)
    P = len(n_agents)
    plain = np.zeros(P, dtype=np.int64)
    size = L.lib.fo_agent_batch_layout(P, n_agents.ctypes.data, t_stride.ctypes.data, plain.ctypes.data)
    off = np.zeros(P, dtype=np.int64)
    zero = np.zeros(P, dtype=np.uint8)
    assert L.lib.fo_agent_batch_layout_corr(P, n_agents.ctypes.data, t_stride.ctypes.data, zero.ctypes.data,
                                            off.ctypes.data) == size
    assert np.array_equal(off, plain)
    corr = np.array([1, 1, 0, 1, 1, 1], dtype=np.uint8)
    size = L.lib.fo_agent_batch_layout_corr(P, n_agents.ctypes.data, t_stride.ctypes.data, corr.ctypes.data,
                                            off.ctypes.data)
    want, o = [], 0
    for a, t, c in zip(n_agents, t_stride, corr):
        want.append(o)
        if a > 0 and t > 0:
            n = L.lib.fo_agent_table_bytes_corr(int(a), int(t)) if c else L.lib.fo_agent_table_bytes(int(a), int(t))
            o += (n + 15) // 16 * 16
    assert list(off) == want and size == o and np.all(off % 16 == 0)
    # malformed: 0 and a message
    assert L.lib.fo_agent_batch_layout_corr(P, n_agents.ctypes.data, t_stride.ctypes.data, None, off.ctypes.data) == 0
    assert b"fo_agent_batch_layout_corr" in L.lib.fo_last_error()
    assert L.lib.fo_agent_batch_layout_corr(-1, None, None, None, None) == 0
    bad = t_stride.copy()
    bad[2] = 129
    assert L.lib.fo_agent_batch_layout_corr(P, n_agents.ctypes.data, bad.ctypes.data, corr.ctypes.data,
                                            off.ctypes.data) == 0
    assert b"problem 2" in L.lib.fo_last_error()
    assert L.lib.fo_agent_batch_layout_corr(0, None, None, None, None) == 0


def test_correlated_entry_points_reject_null_flags_and_vehicles_without_device():
    from frenetix_occlusion_b200 import _lib as L
    fleet, flags = _vehicles(L, 2), _flags(2, 1)
    a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
    for fn in ("fo_metric_batch_corr", "fo_metric_batch_detail_corr"):
        if fn.endswith("detail_corr"):
            a.common.pair = 1 << 24
        assert getattr(L.lib, fn)(C.byref(a), None, fleet, None) == FO_ERR_INVALID_ARG
        assert fn.encode() in L.lib.fo_last_error()
        assert getattr(L.lib, fn)(C.byref(a), flags, None, None) == FO_ERR_INVALID_ARG
        e = _batch_args(L, [], 0)                   # no problems: nothing is read
        e.common.pair = a.common.pair
        assert getattr(L.lib, fn)(C.byref(e), None, None, None) == 0
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = 4, 31
    for f in ("x", "y", "yaw", "v", "var_x", "var_y", "n_states", "kind", "length", "width", "buf_length", "buf_width"):
        setattr(raw, f, 1 << 23)
    pr = (L.FoBatchProblem * 2)()
    pr[0].n_agents, pr[0].t_stride, pr[1].n_agents, pr[1].t_stride, pr[1].table_offset = 2, 31, 2, 31, 16384
    arena, cov = C.c_void_p(1 << 20), C.c_void_p(1 << 22)
    fn = L.lib.fo_agents_pack_batch_corr
    assert fn(C.byref(raw), cov, 2, pr, None, fleet, arena, 1 << 16, None) == FO_ERR_INVALID_ARG
    assert b"fo_agents_pack_batch_corr" in L.lib.fo_last_error()
    assert fn(C.byref(raw), cov, 2, pr, flags, None, arena, 1 << 16, None) == FO_ERR_INVALID_ARG
    # NULL cov_xy with a correlated problem that has agents
    for p in range(2):
        assert fn(C.byref(raw), None, 2, pr, (C.c_uint8 * 2)(*[int(q == p) for q in range(2)]), fleet, arena, 1 << 16,
                  None) == FO_ERR_INVALID_ARG
        assert b"cov_xy" in L.lib.fo_last_error()
    # ... accepted when no correlated problem has agents (here no problem has any: nothing to pack)
    raw.n_agents = 0
    pr[0].n_agents = pr[1].n_agents = 0
    assert fn(C.byref(raw), None, 2, pr, flags, fleet, arena, 1 << 16, None) == 0
    assert fn(C.byref(raw), None, 0, None, None, None, None, 0, None) == 0


def test_a_correlated_table_is_checked_against_its_own_size_without_device():
    """A table that holds a diagonal table of its agents but not the correlated one is outside the arena when flagged."""
    from frenetix_occlusion_b200 import _lib as L
    A, T = 5, 31
    diag, corr = L.lib.fo_agent_table_bytes(A, T), L.lib.fo_agent_table_bytes_corr(A, T)
    assert corr > diag
    arena_bytes = (diag + 15) // 16 * 16
    fleet = _vehicles(L, 1)
    for fn in ("fo_metric_batch_corr", "fo_metric_batch_detail_corr"):
        a = _batch_args(L, [(0, 4, A, T, 0)], 4, arena_bytes=arena_bytes)
        if fn.endswith("detail_corr"):
            a.common.pair = 1 << 24
        assert getattr(L.lib, fn)(C.byref(a), _flags(1, 1), fleet, None) == FO_ERR_INVALID_ARG, fn
        assert b"correlated table of problem 0" in L.lib.fo_last_error()
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = A, T
    pr = (L.FoBatchProblem * 1)()
    pr[0].n_agents, pr[0].t_stride = A, T
    assert L.lib.fo_agents_pack_batch_corr(C.byref(raw), C.c_void_p(1 << 22), 1, pr, _flags(1, 1), fleet,
                                           C.c_void_p(1 << 20), arena_bytes, None) == FO_ERR_INVALID_ARG
    assert b"correlated table of problem 0" in L.lib.fo_last_error()


def test_correlated_entry_points_validate_like_their_diagonal_counterparts_without_device():
    from frenetix_occlusion_b200 import _lib as L
    fleet = _vehicles(L, 8)
    for fn, cases in (("fo_metric_batch_vehicles", _malformed_summary_cases(L)),
                      ("fo_metric_batch_detail_vehicles", _malformed_detail_cases(L))):
        new_fn = fn.replace("_vehicles", "_corr")
        for name, a in cases:
            old = getattr(L.lib, fn)(C.byref(a), fleet, None)
            for flag in (0, 1):
                new = getattr(L.lib, new_fn)(C.byref(a), _flags(8, flag), fleet, None)
                assert old != 0 and new == old, (fn, name, flag, old, new)
                assert new_fn.encode() in L.lib.fo_last_error(), (fn, name)
    # peer stores stay on the single-problem summary path
    for fn in ("fo_metric_batch_corr", "fo_metric_batch_detail_corr"):
        a = _batch_args(L, [(0, 4, 2, 31, 0)], 4)
        a.common.n_peers = 1
        if fn.endswith("detail_corr"):
            a.common.pair = 1 << 24
        assert getattr(L.lib, fn)(C.byref(a), _flags(1, 1), fleet, None) == FO_ERR_UNSUPPORTED, fn
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = 3, 31
    pr = (L.FoBatchProblem * 2)()
    pr[0].n_agents, pr[0].t_stride, pr[1].n_agents, pr[1].t_stride, pr[1].table_offset = 2, 31, 2, 31, 16384
    arena, cov = C.c_void_p(1 << 20), C.c_void_p(1 << 22)
    for n_agents, arena_bytes, r in ((3, 1 << 16, raw), (4, 8192, raw), (4, 1 << 16, raw), (4, 1 << 16, None)):
        raw.n_agents = n_agents
        rp = C.byref(r) if r is not None else None
        old = L.lib.fo_agents_pack_batch_vehicles(rp, 2, pr, fleet, arena, arena_bytes, None)
        for flag in (0, 1):
            new = L.lib.fo_agents_pack_batch_corr(rp, cov, 2, pr, _flags(2, flag), fleet, arena, arena_bytes, None)
            assert old == FO_ERR_INVALID_ARG and new == old, (n_agents, arena_bytes, flag, old, new)


def test_batched_correlated_kernels_stay_inside_their_code_size_budgets():
    """Budgets: the sizes measured when the kernels were added (DESIGN.md 5.11) plus 4 kB."""
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
    budget = {("fo_metric_batch_corr_kernel", "ILb1ELb0E"): 72.25,    # one-warp window-filter shape
              ("fo_metric_batch_corr_kernel", "ILb1ELb1E"): 85.375,   # ... with the float64 tie path
              ("fo_metric_batch_corr_kernel", "ILb0ELb0E"): 83.125,   # team shape
              ("fo_metric_batch_corr_kernel", "ILb0ELb1E"): 99.125,
              ("fo_metric_batch_detail_corr_kernel",): 78.625}
    for parts, kb in budget.items():
        assert size_of(*parts) <= (kb + 4) * 1024, (parts, size_of(*parts))


# ---------------------------------------------------------------------------------------------------- GPU
def _correlate(problem, seed):
    """The problem with correlated covariances (corr_oracle.add_correlations) on every agent; positions unchanged."""
    from frenetix_occlusion_b200.engine import AgentSet
    ag, origin, ego, case = problem
    if ag.n_agents == 0:
        return problem
    case = CO.add_correlations(copy.deepcopy(case), seed)
    c = AgentSet.from_case(case["agents"])
    ag = copy.copy(ag)
    ag.var_x, ag.var_y, ag.cov_xy = c.var_x, c.var_y, c.cov_xy
    assert ag.cov_xy is not None
    return ag, origin, ego, case


def _mixed(seed, T, a_set=(0, 1, 5, 17, 40, 300), n_set=(0, 1, 64, 500), n_problems=16, metrics=None,
           thresholds=None, every=2, varied=False):
    """test_metric_batch._problems with one vehicle each; every `every`-th problem (from the first) correlated, none for
    every = 0."""
    probs = _problems(seed, T, n_problems=n_problems, a_set=list(a_set), n_set=list(n_set), metrics=metrics,
                      thresholds=thresholds, varied=varied)
    probs = [_correlate(p, seed * 100 + i) if every and i % every == 0 else p for i, p in enumerate(probs)]
    return probs, _fleet(len(probs), seed)


def _single(case, veh, ag, origin, ego, want_pair=False, want_step=False):
    single = _engine(case, veh)
    single.set_agents(ag, origin=origin)
    assert single._corr == (ag.cov_xy is not None and ag.n_agents > 0)
    return single.assess(ego, want_pair=want_pair, want_step=want_step)


def _assert_mixed_batch_equals_single(probs, fleet, want_pair=False, want_step=False):
    import torch
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet, correlated=True)
    assert eng._batch["corr"].any()
    parts = eng.assess_batch([p[2] for p in probs], want_pair=want_pair, want_step=want_step).split()
    fields = ("valid", "flags", "summary") + (("pair",) if want_pair else ()) + (("step",) if want_step else ())
    for i, ((ag, origin, ego, case), veh, got) in enumerate(zip(probs, fleet, parts)):
        if not len(ego):
            assert got.valid.numel() == 0
            continue
        want = _single(case, veh, ag, origin, ego, want_pair, want_step)
        torch.cuda.synchronize()
        for f in fields:
            _assert_equal(getattr(got, f), getattr(want, f), (i, f, ag.n_agents, len(ego), ag.cov_xy is not None))
    return parts


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("warps", [1, 4])
def test_mixed_batch_equals_single_problem_path(T, warps, cuda_device, monkeypatch):
    """W = 1 puts both shape classes of both covariance kinds into one call (four launches); W = 4 the team shape."""
    monkeypatch.setenv("FO_TEAM_WARPS", str(warps))
    probs, fleet = _mixed(T + 400, T)
    assert {p[0].n_agents for p in probs} == {0, 1, 5, 17, 40, 300} and {len(p[2]) for p in probs} == {0, 1, 64, 500}
    kinds = {(p[0].n_agents >= 17, p[0].cov_xy is not None) for p in probs if len(p[2]) and p[0].n_agents}
    assert kinds == {(False, False), (False, True), (True, False), (True, True)}
    _assert_mixed_batch_equals_single(probs, fleet)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("detail", ["pair", "step", "both"])
def test_mixed_detail_batch_equals_single_problem_path(T, detail, cuda_device):
    probs, fleet = _mixed(T + 500, T)
    _assert_mixed_batch_equals_single(probs, fleet, detail != "step", detail != "pair")


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["correlated first", "diagonal first"])
def test_detail_batch_with_correlated_problems_between_diagonal_ones(order, cuda_device):
    """The diagonal launch covers the rows of the correlated problems before its last problem (as problems without
    agents) and the correlated launch writes them again: runs of either kind at both ends of the batch."""
    probs, fleet = _mixed(61, 31, a_set=(3, 40, 17, 5), n_set=(64, 1, 200), n_problems=9,
                          every=2 if order == "correlated first" else 3)
    if order == "diagonal first":
        probs = probs[1:] + probs[:1]
        fleet = fleet[1:] + fleet[:1]
    _assert_mixed_batch_equals_single(probs, fleet, True, True)


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", [None, "default", ["dce", "ttc", "wttc"], ["ttc", "be", "hr", "cp"]])
@pytest.mark.parametrize("armed", [False, True])
@pytest.mark.parametrize("detail", [False, True])
def test_mixed_batch_equals_single_problem_path_metrics_and_thresholds(metrics, armed, detail, cuda_device,
                                                                       monkeypatch):
    """Armed dce / ttc / be thresholds run the float64 rounding-tie variants of both covariance kinds."""
    from frenetix_occlusion_b200 import synthetic as S
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    m = S.DEFAULT_METRICS if metrics == "default" else metrics
    thr = dict(S.DEFAULT_THRESHOLDS, dce=0.5, ttc=1.5, be=0.8) if armed else None
    probs, fleet = _mixed(71 + armed, 31, metrics=m, thresholds=thr, n_set=(0, 1, 64, 200), n_problems=12)
    _assert_mixed_batch_equals_single(probs, fleet, detail, detail)


@pytest.mark.gpu
def test_mixed_batch_tables_are_byte_identical_to_single_packs(cuda_device):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    probs, fleet = _mixed(73, 51, n_set=(1,), every=3)
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet, correlated=True)
    arena = eng._batch["arena"]
    n_corr = 0
    for p, ((ag, origin, _, case), veh) in enumerate(zip(probs, fleet)):
        if ag.n_agents == 0:
            continue
        single = _engine(case, veh)
        single.set_agents(ag, origin=origin)
        corr = ag.cov_xy is not None
        n_corr += corr
        assert bool(eng._batch["corr"][p]) == corr
        off = eng._batch["problems"][p].table_offset
        n = L.lib.fo_agent_table_bytes(ag.n_agents, ag.t_stride)
        torch.cuda.synchronize()
        assert torch.equal(arena[off:off + n], single._table[:n]), p
        if corr:                                         # the s3 section behind the diagonal table's 16-byte padding
            lo, hi = (n + 15) // 16 * 16, L.lib.fo_agent_table_bytes_corr(ag.n_agents, ag.t_stride)
            assert single._table.numel() == hi and torch.equal(arena[off + lo:off + hi], single._table[lo:hi]), p
    assert n_corr >= 3


class _Recorder:
    """Stands in for the ctypes library and records the names of the entry points called through it."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        self.calls.append(name)
        return getattr(self._lib, name)


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_all_diagonal_batch_with_correlated_allowed_makes_the_diagonal_launches(detail, cuda_device, monkeypatch):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    probs, fleet = _mixed(79, 31, n_set=(1, 64), n_problems=8, every=0)

    def run(correlated):
        rec = _Recorder(L.lib)
        monkeypatch.setattr(L, "lib", rec)
        eng = _engine(probs[0][3])
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet, correlated=correlated)
            got = eng.assess_batch([p[2] for p in probs], want_pair=detail, want_step=detail)
            torch.cuda.synchronize()
        monkeypatch.setattr(L, "lib", rec._lib)
        assert not eng._batch["corr"].any()
        kernels = [e.name for e in sorted(prof.events(), key=lambda e: e.time_range.start)
                   if e.device_type == torch.autograd.DeviceType.CUDA and "fo::" in e.name]
        return [c for c in rec.calls if c.startswith("fo_") and c not in ("fo_last_error",)], kernels, got
    calls_c, kernels_c, got_c = run(True)
    calls_d, kernels_d, got_d = run(False)
    assert calls_c == calls_d
    assert calls_c == ["fo_agent_batch_layout_corr", "fo_agents_pack_batch_corr",
                       "fo_metric_batch_detail_corr" if detail else "fo_metric_batch_corr"]
    # with every flag 0 the _corr calls make the launches of the diagonal ones: no correlated kernel runs
    assert kernels_c == kernels_d
    assert kernels_c and not any("corr" in k for k in kernels_c), kernels_c
    assert any(("fo_metric_batch_detail_kernel" if detail else "fo_metric_batch_kernel") in k for k in kernels_c), kernels_c
    for f in ("valid", "flags", "summary") + (("pair", "step") if detail else ()):
        _assert_equal(getattr(got_c, f), getattr(got_d, f), f)
    for (ag, origin, ego, case), veh, g in zip(probs, fleet, got_c.split()):
        if len(ego):
            want = _single(case, veh, ag, origin, ego, detail, detail)
            for f in ("valid", "flags", "summary") + (("pair", "step") if detail else ()):
                _assert_equal(getattr(g, f), getattr(want, f), f)


@pytest.mark.gpu
def test_two_problems_of_a_mixed_batch_match_the_oracle(cuda_device, monkeypatch):
    from test_metric_corr import _check
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    probs, fleet = _mixed(83, 31, a_set=(5, 40), n_set=(80, 60), n_problems=2)
    assert probs[0][0].cov_xy is not None and probs[1][0].cov_xy is None
    for detail in (False, True):
        eng = _engine(probs[0][3])
        eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet, correlated=True)
        parts = eng.assess_batch([p[2] for p in probs], want_pair=detail, want_step=detail).split()
        for (ag, origin, ego, case), veh, got in zip(probs, fleet, parts):
            # the oracle runs in the problem's own frame: the same float64 shift the batch applies
            sub = dict(case, vehicle=dict(veh), agents=[dict(a) for a in case["agents"]])
            for a, k in zip(sub["agents"], range(ag.n_agents)):
                n = int(ag.n_states[k])
                a["pos"] = np.stack((ag.x[k, :n] - origin[0], ag.y[k, :n] - origin[1]), -1).astype(np.float32).astype(np.float64)
            sub["ego"] = (ego - np.array([origin[0], origin[1], 0, 0, 0])).astype(np.float32).astype(np.float64)
            out = CO.evaluate_bundle(sub)
            res = {"valid": got.valid.cpu().numpy(), "summary": got.summary.cpu().numpy(),
                   "flags": got.flags.cpu().numpy().astype(np.uint32)}
            if detail:
                res["pair"], res["step"] = got.pair.cpu().numpy(), got.step.cpu().numpy()
            _check(parity.compare_bundle(out, res, sub))


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_a_covariance_that_is_not_positive_definite_stays_in_its_problem(detail, cuda_device, monkeypatch):
    """|rho| = 1.5 on one agent of one problem, set on the AgentSet after its validation: that problem gets NaN
    collision probabilities, as alone, and every other problem its single-path outputs."""
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    probs, fleet = _mixed(89, 31, a_set=(20, 5, 40, 3), n_set=(120, 64), n_problems=6, metrics=["cp", "hr"])
    case = S.make_case(120, 20, 31, seed=89, activated_metrics=["cp", "hr"])
    for a in case["agents"]:
        a["pos"] = np.asarray(a["pos"]) * 0.3            # onto the ego paths: many gated steps
    ag = AgentSet.from_case(case["agents"])
    ag.cov_xy = np.zeros_like(ag.var_x)
    ag.cov_xy[0] = 1.5 * np.sqrt(ag.var_x[0] * ag.var_y[0])
    probs[2] = (ag, (0.0, 0.0), case["ego"], case)
    parts = _assert_mixed_batch_equals_single(probs, fleet, detail, detail)
    # NaN where fo_metric_bundle_corr puts it: the per-step CP of the detail path, max_collision_probability_all of the
    # summary path
    nan_cp = (lambda g: np.isnan(g.step.cpu().numpy()[..., 0])) if detail else \
        (lambda g: np.isnan(g.summary.cpu().numpy()[:, 4]))
    assert nan_cp(parts[2]).any()
    if detail:
        assert np.isfinite(parts[2].step.cpu().numpy()[:, 1:, :, 0]).all()
    for i, g in enumerate(parts):
        if i != 2 and g.valid.numel():
            assert not nan_cp(g).any(), i


# ---- interfaces whose predictions carry correlated covariances --------------------------------------------------
def _align_covariances(fo):
    """cov_list of every prediction = R(theta) diag(2 var, 0.5 var) R(theta)^T of its orientation: longer along the
    heading than across it (var: the prediction's own variance)."""
    for pred in fo.agent_manager.predictions.values():
        cov = np.asarray(pred["cov_list"], dtype=np.float64)
        th = np.asarray(pred["orientation_list"], dtype=np.float64)[:len(cov)]
        c, s = np.cos(th), np.sin(th)
        lo, la = 2.0 * cov[:, 0, 0], 0.5 * cov[:, 0, 0]
        out = np.empty_like(cov)
        out[:, 0, 0] = c * c * lo + s * s * la
        out[:, 1, 1] = s * s * lo + c * c * la
        out[:, 0, 1] = out[:, 1, 0] = c * s * (lo - la)
        pred["cov_list"] = out


def _corr_scenes():
    fleet = _fleet(len(SCENES), 97)
    pairs = [_scene_interface_with(n, v) for n, v in zip(SCENES, fleet)]
    fos = [p[0] for p in pairs]
    for fo in fos[::2]:
        _align_covariances(fo)
    return fos, [p[1] for p in pairs]


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_assess_interfaces_with_correlated_predictions_equals_each_interface(detail, cuda_device, monkeypatch):
    import torch
    from frenetix_occlusion_b200.batch import assess_interfaces
    monkeypatch.setenv("FO_TEAM_WARPS", "1")
    fos, fans = _corr_scenes()
    got = assess_interfaces(fos, fans, want_pair=detail, want_step=detail)
    corr = []
    for i, (fo, fan, g) in enumerate(zip(fos, fans, got)):
        want = fo.assess_bundle(fan, detail, detail)
        torch.cuda.synchronize()
        corr.append(fo.metrics._core.engine._corr)
        for f in ("valid", "flags", "summary") + (("pair", "step") if detail else ()):
            _assert_equal(getattr(g, f), getattr(want, f), (i, f))
    assert any(corr) and not all(corr), corr         # both kinds in the batch


@pytest.mark.gpu
def test_prefetch_interfaces_with_correlated_predictions_serves_every_candidate_like_each_interface(cuda_device):
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.batch import prefetch_interfaces
    fos, fans = _corr_scenes()
    cands = [_trajectories(f) for f in fans]
    l0 = L.lib.fo_launch_count()
    counts = prefetch_interfaces(fos, cands)
    # three pack launches (order, pack, correlation sections) and one detail launch per covariance kind
    assert L.lib.fo_launch_count() - l0 == 5
    assert counts == [len(c) for c in cands]
    l0 = L.lib.fo_launch_count()
    served = [[fo.trajectory_safety_assessment(t) for t in c] for fo, c in zip(fos, cands)]
    assert L.lib.fo_launch_count() == l0, "prefetched trajectories must not launch again"
    for fo, c, s in zip(fos, cands, served):
        fo.metrics._core._fingerprint = None            # the interface's own path from scratch: sync, pack, prefetch
        assert fo.prefetch_assessments(c) == len(c)
        _assert_same_assessments(s, [fo.trajectory_safety_assessment(t) for t in c])
