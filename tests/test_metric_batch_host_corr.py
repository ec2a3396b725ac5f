"""Batches with correlated prediction covariances from host memory in one call (fo_metric_batch_host_corr): float64 ego
rows in the caller's world frame, one float64 origin per problem, float32 cov_xy rows and one flag per problem in, host
arrays out.  The CPU part checks that malformed arguments and covariances that are not positive definite are rejected
before any device work; the GPU part checks that the results equal, bit for bit, MetricEngine.set_agent_batch(
correlated=True) + assess_batch on the same host bundles, fo_metric_batch_host without flags, and set_agents + assess
for a single problem."""
import copy
import ctypes as C

import numpy as np
import pytest

import corr_oracle as CO
import parity
from test_metric_batch import _problems
from test_metric_batch_host import _assert_same, _mix, _params, _pinned, _raw_host, batch_host
from test_metric_batch_vehicles import _fleet

FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2


def _cov_host(agent_sets, n_agents, t_stride, alloc=np.zeros):
    """cov_xy of all problems as fo_metric_batch_host_corr takes it: [A, S] float32, rows aligned with _raw_host's."""
    A, S = int(n_agents.sum()), int(t_stride.max(initial=0))
    cov = alloc((A, S), np.float32)
    a0 = 0
    for ag, n, tp in zip(agent_sets, n_agents, t_stride):
        if n and ag.cov_xy is not None:
            cov[a0:a0 + n, :tp] = ag.cov_xy
        a0 += int(n)
    return cov


def _call(L, params, agent_sets, origins, egos, vehicles=None, corr=None, want_pair=False, want_step=False,
          pinned=False, cov_null=False):
    """fo_metric_batch_host_corr on host copies of the problems, as a ctypes embedder calls it.  corr: the flags (default:
    the sets with cov_xy).  Returns the status and the host outputs."""
    from frenetix_occlusion_b200.engine import vehicle_struct
    P = len(agent_sets)
    alloc = (lambda shape, dtype: _pinned(shape, dtype)) if pinned else np.zeros
    org = alloc((P, 2), np.float64)
    org[:] = np.asarray(origins, dtype=np.float64).reshape(P, 2)
    raw, n_agents, t_stride = _raw_host(L, agent_sets, org, alloc)
    cov = _cov_host(agent_sets, n_agents, t_stride, alloc)
    flags = np.array([a.cov_xy is not None for a in agent_sets] if corr is None else corr, dtype=np.uint8)
    T = int(egos[0].shape[1])
    counts = np.array([len(e) for e in egos], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    N = int(offsets[-1])
    ego = alloc((N, T, 5), np.float64)
    for p, e in enumerate(egos):
        ego[offsets[p]:offsets[p + 1]] = e
    problems = (L.FoBatchProblem * max(P, 1))()
    for p in range(P):
        problems[p].traj_begin, problems[p].n_traj = int(offsets[p]), int(counts[p])
        problems[p].n_agents, problems[p].t_stride = int(n_agents[p]), int(t_stride[p])
    veh = (L.FoVehicle * max(P, 1))(*[vehicle_struct(v) for v in vehicles]) if vehicles is not None else None
    pairs = int(np.dot(counts, n_agents))
    out = {"valid": np.empty(N, np.uint8), "flags": np.empty(N, np.uint32),
           "summary": np.empty((N, L.FO_SUMMARY_K), np.float32)}
    if want_pair:
        out["pair"] = np.full(pairs * L.FO_PAIR_K, -7.0, np.float32)
    if want_step:
        out["step"] = np.full(pairs * max(T - 1, 0) * L.FO_STEP_K, -7.0, np.float32)
    ptr = lambda k: out[k].ctypes.data if k in out else None  # noqa: E731
    rc = L.lib.fo_metric_batch_host_corr(ego.ctypes.data, N, T, org.ctypes.data, C.byref(raw),
                                         None if cov_null else cov.ctypes.data, P, problems, flags.ctypes.data, veh,
                                         C.byref(params), ptr("valid"), ptr("summary"), ptr("flags"), ptr("pair"),
                                         ptr("step"))
    return rc, out


def batch_host_corr(eng, agent_sets, origins, egos, **kw):
    from frenetix_occlusion_b200 import _lib as L
    rc, out = _call(L, _params(eng), agent_sets, origins, egos, **kw)
    L.check(rc, "fo_metric_batch_host_corr")
    return out


def engine_batch_corr(eng, agent_sets, origins, egos, vehicles=None, want_pair=False, want_step=False):
    """The same through the Python batch path (set_agent_batch(correlated=True) + assess_batch), copied to the host."""
    eng.set_agent_batch(agent_sets, origins, vehicles=vehicles, correlated=True)
    r = eng.assess_batch(egos, want_pair=want_pair, want_step=want_step)
    out = {"valid": r.valid.cpu().numpy(), "flags": r.flags.cpu().numpy().view(np.uint32),
           "summary": r.summary.cpu().numpy()}
    if want_pair:
        out["pair"] = r.pair.cpu().numpy()
    if want_step:
        out["step"] = r.step.cpu().numpy()
    return out


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


def _corr_mix(seed, T, which="half", **kw):
    """test_metric_batch_host._mix (UTM-sized coordinates) with all / every other / none of the problems correlated."""
    probs = _mix(seed, T, **kw)
    every = {"all": 1, "half": 2, "none": 0}[which]
    return [_correlate(p, seed * 100 + i) if every and i % every == 0 else p for i, p in enumerate(probs)]


def _engine(case):
    from frenetix_occlusion_b200.engine import MetricEngine
    return MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])


def _assert_host_corr_equals_engine(probs, vehicles=None, want_pair=False, want_step=False, pinned=False, eng=None):
    eng = eng or _engine(probs[0][3])
    args = ([p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs])
    got = batch_host_corr(eng, *args, vehicles=vehicles, want_pair=want_pair, want_step=want_step, pinned=pinned)
    want = engine_batch_corr(eng, *args, vehicles=vehicles, want_pair=want_pair, want_step=want_step)
    _assert_same(got, want)
    return got


# ---------------------------------------------------------------------------------------------------- CPU
def _cpu_params(L):
    a = L.FoMetricArgs()
    a.vehicle = L.FoVehicle(4.5, 1.6, 1200.0, 1.4, 10.0)
    a.dt, a.metric_mask = 0.1, 0x7f
    return a


def _cpu_batch(seed=5):
    """Three small problems (2, 0 and 3 agents; the third correlated) whose arguments are valid: what is rejected below
    is rejected for the one thing each case changes, before the library touches the device."""
    probs = _problems(seed, 31, n_problems=3, a_set=[2, 0, 3], n_set=[4])
    probs[2] = _correlate(probs[2], seed)
    return [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs]


def _corr_desc_call(L, problems, n_traj, T=31, flags=1, raw_stride=31, fn="fo_metric_batch_host_corr", **common):
    """The host entry points on descriptors (traj_begin, n_traj, n_agents, t_stride, table_offset) with host buffers
    that are never read."""
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p)
    arr = (L.FoBatchProblem * max(len(problems), 1))()
    for i, (b, n, na, tp, off) in enumerate(problems):
        arr[i].traj_begin, arr[i].n_traj, arr[i].n_agents, arr[i].t_stride, arr[i].table_offset = b, n, na, tp, off
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = sum(q[2] for q in problems), raw_stride
    for f, _ in L.FoAgentsRaw._fields_[2:]:
        setattr(raw, f, p.value)
    a = L.FoMetricArgs()
    a.metric_mask = 0x7f
    for k, v in common.items():
        setattr(a, k, v)
    corr = (C.c_uint8 * max(len(problems), 1))(*([flags] * len(problems)))
    if fn == "fo_metric_batch_host":
        return L.lib.fo_metric_batch_host(p, n_traj, T, p, C.byref(raw), len(problems), arr, None, C.byref(a), p, p, p,
                                          None, None)
    return L.lib.fo_metric_batch_host_corr(p, n_traj, T, p, C.byref(raw), p, len(problems), arr, corr, None, C.byref(a),
                                           p, p, p, None, None)


def test_batch_host_corr_rejects_null_flags_and_covariances_without_device():
    from frenetix_occlusion_b200 import _lib as L
    ags, origins, egos = _cpu_batch()
    params = _cpu_params(L)
    # NULL corr_host with problems
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    raw = L.FoAgentsRaw()
    pr = (L.FoBatchProblem * 1)()
    assert L.lib.fo_metric_batch_host_corr(p, 0, 31, p, C.byref(raw), None, 1, pr, None, None, C.byref(params), p, None,
                                           None, None, None) == FO_ERR_INVALID_ARG
    assert b"fo_metric_batch_host_corr: corr_host" in L.lib.fo_last_error()
    # NULL cov_xy with a flagged problem that has agents ...
    rc, _ = _call(L, params, ags, origins, egos, cov_null=True)
    assert rc == FO_ERR_INVALID_ARG and b"cov_xy" in L.lib.fo_last_error()
    rc, _ = _call(L, params, ags, origins, egos, corr=[1, 0, 0], cov_null=True)
    assert rc == FO_ERR_INVALID_ARG and b"problem 0" in L.lib.fo_last_error()
    # ... but not with a flag on a problem without agents only (no trajectories: nothing reaches the device)
    rc, _ = _call(L, params, ags, origins, [e[:0] for e in egos], corr=[0, 1, 0], cov_null=True)
    assert rc == 0
    # nothing to do
    assert L.lib.fo_metric_batch_host_corr(None, 0, 31, None, None, None, 0, None, None, None, C.byref(params), None,
                                           None, None, None, None) == 0


def test_batch_host_corr_rejects_peers_and_malformed_batches_without_device():
    from frenetix_occlusion_b200 import _lib as L
    ok = [(0, 4, 2, 31, 0), (4, 3, 1, 31, 0)]
    for flag in (0, 1):
        assert _corr_desc_call(L, ok, 7, flags=flag, n_peers=1) == FO_ERR_UNSUPPORTED
        assert b"fo_metric_batch_host_corr" in L.lib.fo_last_error()
    # the statuses fo_metric_batch_host gives the same descriptors, with this call's name in the message
    for name, pr, n, T in (("gap", [(0, 4, 2, 31, 0), (5, 3, 2, 31, 0)], 8, 31),
                           ("order", [(4, 3, 2, 31, 0), (0, 4, 2, 31, 0)], 7, 31),
                           ("uncovered", [(0, 4, 2, 31, 0)], 6, 31),
                           ("t_stride", [(0, 4, 2, 129, 0)], 4, 31),
                           ("T", [(0, 4, 2, 31, 0)], 4, 129)):
        old = _corr_desc_call(L, pr, n, T, raw_stride=129, fn="fo_metric_batch_host")
        for flag in (0, 1):
            new = _corr_desc_call(L, pr, n, T, flags=flag, raw_stride=129)
            assert old < 0 and new == old, (name, flag, old, new)
            assert b"fo_metric_batch_host_corr" in L.lib.fo_last_error(), name
    assert _corr_desc_call(L, [(0, 4, 2, 51, 0)], 4, raw_stride=31) == FO_ERR_INVALID_ARG     # row stride too small


@pytest.mark.parametrize("case", ["|rho| >= 1", "zero variance, covariance", "one zero variance"])
def test_batch_host_corr_rejects_covariances_that_are_not_positive_definite_without_device(case):
    """Problem 2, agent 1, state 8 reads covariance 7; the message names them.  The last case passes the reference's
    diagonal rule (no correlation there) but has rho = 0 / 0 on the correlated path."""
    from frenetix_occlusion_b200 import _lib as L
    ags, origins, egos = _cpu_batch()
    ag = ags[2] = copy.copy(ags[2])
    ag.var_x, ag.var_y, ag.cov_xy = ag.var_x.copy(), ag.var_y.copy(), ag.cov_xy.copy()
    if case == "|rho| >= 1":
        ag.cov_xy[1, 7] = 1.0001 * np.sqrt(ag.var_x[1, 7] * ag.var_y[1, 7])
    elif case == "zero variance, covariance":
        ag.var_x[1, 7] = 0.0
    else:
        ag.var_y[1, 7], ag.cov_xy[1, 7] = 0.0, 0.0
    rc, _ = _call(L, _cpu_params(L), ags, origins, egos)
    assert rc == FO_ERR_INVALID_ARG
    assert L.lib.fo_last_error() == (b"fo_metric_batch_host_corr: problem 2, agent 1: covariance 7 is not positive "
                                     b"definite")
    # the same covariance in a problem that is not flagged is never read
    ags[2] = copy.copy(ag)
    rc, _ = _call(L, _cpu_params(L), ags, origins, [e[:0] for e in egos], corr=[0, 0, 0])
    assert rc == 0


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51])
@pytest.mark.parametrize("which", ["all", "half", "none"])
@pytest.mark.parametrize("detail", [False, True])
@pytest.mark.parametrize("warps", [None, "1"])
def test_batch_host_corr_equals_the_engine_batch(T, which, detail, warps, cuda_device, monkeypatch):
    """Agent counts 0-300 and trajectory counts 0-500 (W = 1 runs both shapes of both covariance kinds), every problem
    at UTM-sized coordinates and with its own vehicle."""
    if warps:
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
    else:
        monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    probs = _corr_mix(T + 600, T, which)
    assert {p[0].n_agents for p in probs} == {0, 1, 3, 16, 17, 33, 300} and {len(p[2]) for p in probs} == {0, 1, 64, 500}
    n_corr = sum(p[0].cov_xy is not None for p in probs)
    assert (n_corr == 0) == (which == "none") and (n_corr < len(probs) - 2) == (which != "all")
    _assert_host_corr_equals_engine(probs, _fleet(len(probs), T), detail, detail)


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", ["default", "all"])
@pytest.mark.parametrize("armed", [False, True])
@pytest.mark.parametrize("detail", [False, True])
@pytest.mark.parametrize("warps", [None, "1"])
def test_batch_host_corr_equals_the_engine_batch_metrics_and_thresholds(metrics, armed, detail, warps, cuda_device,
                                                                        monkeypatch):
    """Armed dce / ttc / be thresholds run the float64 rounding-tie variants of both covariance kinds."""
    from frenetix_occlusion_b200 import synthetic as S
    if warps:
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
    else:
        monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    m = S.DEFAULT_METRICS if metrics == "default" else S.ALL_METRICS
    thr = dict(S.DEFAULT_THRESHOLDS, dce=0.5, ttc=1.5, be=0.8) if armed else None
    probs = _corr_mix(97 + armed, 31, metrics=m, thresholds=thr, n_set=(0, 1, 64, 200))
    _assert_host_corr_equals_engine(probs, None, detail, detail)


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_batch_host_corr_without_flags_equals_batch_host(detail, cuda_device):
    """Correlated sets, no flag set: the diagonal variances only, as fo_metric_batch_host gives them."""
    from frenetix_occlusion_b200 import _lib as L
    probs = _corr_mix(101, 31, "all")
    eng = _engine(probs[0][3])
    args = ([p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs])
    fleet = _fleet(len(probs), 101)
    rc, got = _call(L, _params(eng), *args, vehicles=fleet, corr=[0] * len(probs), want_pair=detail, want_step=detail)
    L.check(rc, "fo_metric_batch_host_corr")
    diag = [copy.copy(a) for a in args[0]]
    for a in diag:
        a.cov_xy = None
    want = batch_host(eng, diag, args[1], args[2], vehicles=fleet, want_pair=detail, want_step=detail)
    _assert_same(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 5, 17, 40, 300])
@pytest.mark.parametrize("detail", [False, True])
def test_one_correlated_problem_equals_the_single_path(A, detail, cuda_device, monkeypatch):
    """n_problems = 1 is the correlated single planner: fo_agents_pack_corr + fo_metric_bundle_corr bit for bit, with the
    team size the library picks."""
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    probs = _corr_mix(103 + A, 31, "all", a_set=(A,), n_set=(700,), n_problems=1)
    ag, origin, ego, case = probs[0]
    assert ag.cov_xy is not None
    eng = _engine(case)
    got = batch_host_corr(eng, [ag], [origin], [ego], want_pair=detail, want_step=detail)
    single = _engine(case)
    single.set_agents(ag, origin=origin)
    assert single._corr
    r = single.assess(ego, want_pair=detail, want_step=detail)
    want = {"valid": r.valid.cpu().numpy(), "flags": r.flags.cpu().numpy().view(np.uint32),
            "summary": r.summary.cpu().numpy()}
    if detail:
        want["pair"], want["step"] = r.pair.cpu().numpy().ravel(), r.step.cpu().numpy().ravel()
    _assert_same(got, want)


@pytest.mark.gpu
def test_two_problems_of_a_correlated_host_batch_match_the_oracle(cuda_device):
    from test_metric_corr import _check
    probs = _corr_mix(107, 31, "all", a_set=(5, 17), n_set=(60, 40), n_problems=2)
    assert all(p[0].cov_xy is not None for p in probs)
    assert all(abs(c) > 9e4 for p in probs for c in p[1])             # UTM-sized origins
    fleet = _fleet(2, 107)
    eng = _engine(probs[0][3])
    got = batch_host_corr(eng, [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs], vehicles=fleet,
                          want_pair=True, want_step=True)
    row = q = 0
    for (ag, origin, ego, case), veh in zip(probs, fleet):
        n, a, T = len(ego), ag.n_agents, ego.shape[1]
        # the oracle runs in the problem's own frame: the same float64 shift, then float32
        sub = dict(case, vehicle=dict(veh), agents=[dict(x) for x in case["agents"]])
        for x, k in zip(sub["agents"], range(a)):
            m = int(ag.n_states[k])
            x["pos"] = np.stack((ag.x[k, :m] - origin[0], ag.y[k, :m] - origin[1]), -1).astype(np.float32).astype(np.float64)
        sub["ego"] = (ego - np.array([origin[0], origin[1], 0, 0, 0])).astype(np.float32).astype(np.float64)
        out = CO.evaluate_bundle(sub)
        res = {"valid": got["valid"][row:row + n], "summary": got["summary"][row:row + n],
               "flags": got["flags"][row:row + n],
               "pair": got["pair"][q * 12:(q + n * a) * 12].reshape(n, a, 12),
               "step": got["step"][q * (T - 1) * 3:(q + n * a) * (T - 1) * 3].reshape(n, a, T - 1, 3)}
        _check(parity.compare_bundle(out, res, sub))
        row, q = row + n, q + n * a


def _pad(ag, extra):
    """A copy of an AgentSet with `extra` more columns of padding behind every prediction."""
    out = copy.copy(ag)
    for f in ("x", "y", "yaw", "v", "var_x", "var_y", "cov_xy"):
        setattr(out, f, np.pad(getattr(ag, f), ((0, 0), (0, extra))))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("detail", [False, True])
def test_covariances_the_pack_never_reads_are_accepted(detail, cuda_device):
    """Covariance n_states - 1 and the padding up to t_stride are read by no state: not positive definite there, the
    call is accepted and equals the engine, which never looks at them either."""
    from frenetix_occlusion_b200 import _lib as L
    probs = _corr_mix(109, 31, "all", a_set=(4, 20, 3), n_set=(150, 64, 200), n_problems=3)
    for i in (0, 1):
        ag, origin, ego, case = probs[i]
        ag = _pad(ag, 5)
        ag.var_x, ag.var_y, ag.cov_xy = ag.var_x.copy(), ag.var_y.copy(), ag.cov_xy.copy()
        for k in range(ag.n_agents):
            n = int(ag.n_states[k])
            ag.cov_xy[k, n - 1] = 3.0 * np.sqrt(ag.var_x[k, n - 1] * ag.var_y[k, n - 1])      # |rho| = 3
            ag.cov_xy[k, n:] = 0.5                                                            # zero variances
        probs[i] = (ag, origin, ego, case)
    assert probs[0][0].t_stride == 36
    _assert_host_corr_equals_engine(probs, _fleet(3, 109), detail, detail)
    # one index lower is read (by the last state): rejected before any device work
    ag = probs[1][0]
    ag.cov_xy[2, int(ag.n_states[2]) - 2] = 3.0 * ag.cov_xy[2, int(ag.n_states[2]) - 2] + 1.0
    ag.var_y[2, int(ag.n_states[2]) - 2] = 0.0
    rc, _ = _call(L, _params(_engine(probs[0][3])), [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs])
    assert rc == FO_ERR_INVALID_ARG
    assert f"problem 1, agent 2: covariance {int(ag.n_states[2]) - 2} ".encode() in L.lib.fo_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_batch_host_corr_takes_pageable_and_page_locked_inputs(pinned, cuda_device):
    probs = _corr_mix(113, 51, "half", a_set=(0, 5, 40), n_set=(300, 0, 700), n_problems=6)
    _assert_host_corr_equals_engine(probs, _fleet(len(probs), 113), pinned=pinned)
    _assert_host_corr_equals_engine(probs, None, True, True, pinned=pinned)


@pytest.mark.gpu
def test_diagonal_and_correlated_host_calls_share_one_growing_workspace(cuda_device):
    """fo_metric_batch_host and fo_metric_batch_host_corr in turn on one thread, sizes growing and shrinking: every call
    still equals the engine."""
    from test_metric_batch_host import _assert_host_equals_engine
    small = _corr_mix(127, 31, "half", a_set=(2, 0), n_set=(10, 30), n_problems=2)
    large = _corr_mix(131, 31, "half", a_set=(0, 40, 300, 5), n_set=(500, 800, 64, 1000), n_problems=5)
    larger = _corr_mix(137, 51, "all", a_set=(300, 17, 60), n_set=(1000, 1500, 700), n_problems=3)
    diag = lambda probs: [(_strip(p[0]),) + tuple(p[1:]) for p in probs]  # noqa: E731
    eng = _engine(small[0][3])
    _assert_host_equals_engine(diag(small), eng=eng)
    _assert_host_corr_equals_engine(small, eng=eng)
    _assert_host_corr_equals_engine(large, want_pair=True, want_step=True, eng=eng)
    _assert_host_equals_engine(diag(large), want_pair=True, eng=eng)
    _assert_host_corr_equals_engine(larger, _fleet(3, 137), eng=eng)
    _assert_host_equals_engine(diag(small), want_step=True, eng=eng)
    _assert_host_corr_equals_engine(small, want_step=True, pinned=True, eng=eng)
    _assert_host_equals_engine(diag(larger), _fleet(3, 137), eng=eng)


def _strip(ag):
    out = copy.copy(ag)
    out.cov_xy = None
    return out
