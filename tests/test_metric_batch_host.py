"""Batches of independent planning problems from host memory in one call (fo_metric_batch_host): float64 ego rows in the
caller's world frame and one float64 origin per problem in, host arrays out.  The CPU part checks that every malformed
argument is rejected before any device work, with the status the device batch calls give; the GPU part checks that the
results equal, bit for bit, MetricEngine.set_agent_batch + assess_batch on the same float64 host bundles."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_metric_batch import _batch_args, _problems
from test_metric_batch_vehicles import _fleet

FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _raw_host(L, agent_sets, origins, alloc=np.zeros):
    """The agents of all problems as fo_metric_batch_host takes them: float32 SoA host arrays, concatenated in problem
    order, positions shifted by their problem's origin in float64 -- the buffer set_agent_batch uploads."""
    n_agents = np.array([a.n_agents if a.t_stride > 0 else 0 for a in agent_sets], dtype=np.int32)
    t_stride = np.array([a.t_stride if n else 0 for a, n in zip(agent_sets, n_agents)], dtype=np.int32)
    A, S = int(n_agents.sum()), int(t_stride.max(initial=0))
    fl = alloc((6, A, S), dtype=np.float32)
    pa = alloc((4, A), dtype=np.float32)
    ia = alloc((2, A), dtype=np.int32)
    a0 = 0
    for p, ag in enumerate(agent_sets):
        n, tp = int(n_agents[p]), int(t_stride[p])
        if n == 0:
            continue
        rows = slice(a0, a0 + n)
        fl[0, rows, :tp] = ag.x - origins[p][0]
        fl[1, rows, :tp] = ag.y - origins[p][1]
        fl[2, rows, :tp], fl[3, rows, :tp], fl[4, rows, :tp], fl[5, rows, :tp] = ag.yaw, ag.v, ag.var_x, ag.var_y
        pa[:, rows] = (ag.length, ag.width, ag.buf_length, ag.buf_width)
        ia[:, rows] = (ag.n_states, ag.kind)
        a0 += n
    raw = L.FoAgentsRaw()
    raw.n_agents, raw.t_stride = A, S
    raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y = [fl[i].ctypes.data for i in range(6)]
    raw.length, raw.width, raw.buf_length, raw.buf_width = [pa[i].ctypes.data for i in range(4)]
    raw.n_states, raw.kind = ia[0].ctypes.data, ia[1].ctypes.data
    raw._keep = (fl, pa, ia)
    return raw, n_agents, t_stride


def _pinned(shape, dtype):
    import torch
    t = torch.zeros(shape, dtype={np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32}[dtype])
    return t.pin_memory().numpy()


def _params(eng):
    """The shared configuration of an engine as FoMetricArgs (vehicle, harm, dt, masks, thresholds)."""
    from frenetix_occlusion_b200 import _lib as L
    a = L.FoMetricArgs()
    a.vehicle, a.harm, a.dt = eng.vehicle, eng.harm, eng.dt
    a.metric_mask, a.threshold_mask = eng.metric_mask, eng.threshold_mask
    for name in L.T_BITS:
        v = eng.thresholds.get(name)
        setattr(a, "thr_" + name, float(v) if v is not None else 0.0)
    return a


def batch_host(eng, agent_sets, origins, egos, vehicles=None, want_pair=False, want_step=False, pinned=False):
    """fo_metric_batch_host on host copies of the problems, as a ctypes embedder calls it: returns the host outputs
    (valid, flags, summary, and the flat pair / step arrays where wanted)."""
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.engine import vehicle_struct
    P = len(agent_sets)
    alloc = (lambda shape, dtype: _pinned(shape, dtype)) if pinned else np.zeros
    org = alloc((P, 2), np.float64)
    org[:] = np.asarray(origins, dtype=np.float64).reshape(P, 2)
    raw, n_agents, t_stride = _raw_host(L, agent_sets, org, alloc)
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
    L.check(L.lib.fo_metric_batch_host(ego.ctypes.data, N, T, org.ctypes.data, C.byref(raw), P, problems, veh,
                                       C.byref(_params(eng)), ptr("valid"), ptr("summary"), ptr("flags"), ptr("pair"),
                                       ptr("step")), "fo_metric_batch_host")
    return out


def engine_batch(eng, agent_sets, origins, egos, vehicles=None, want_pair=False, want_step=False):
    """The same through the Python batch path, copied to the host."""
    eng.set_agent_batch(agent_sets, origins, vehicles=vehicles)
    r = eng.assess_batch(egos, want_pair=want_pair, want_step=want_step)
    out = {"valid": r.valid.cpu().numpy(), "flags": r.flags.cpu().numpy().view(np.uint32),
           "summary": r.summary.cpu().numpy()}
    if want_pair:
        out["pair"] = r.pair.cpu().numpy()
    if want_step:
        out["step"] = r.step.cpu().numpy()
    return out


def _assert_same(got, want, what=""):
    assert sorted(got) == sorted(want), what
    for k in want:
        g, w = got[k], want[k]
        assert g.shape == w.shape and g.dtype == w.dtype, (what, k, g.shape, w.shape)
        assert np.array_equal(g, w, equal_nan=True), (what, k)
        if g.dtype.kind == "f":
            assert np.array_equal(np.isnan(g), np.isnan(w)), (what, k)


def _far(probs, seed):
    """The problems of test_metric_batch._problems moved to UTM-sized coordinates: every problem by its own offset of
    1e5-6e6 m (not a float32 value), origins included, so the float64 shift before the rounding matters."""
    rng = np.random.default_rng(seed)
    out = []
    for ag, origin, ego, case in probs:
        dx, dy = rng.uniform(1e5, 6e6, 2)
        ego = ego.astype(np.float64)
        ego[..., 0] += dx
        ego[..., 1] += dy
        live = np.arange(ag.t_stride)[None, :] < ag.n_states[:, None]
        ag.x, ag.y = ag.x + dx * live, ag.y + dy * live
        out.append((ag, (origin[0] + dx, origin[1] + dy), ego, case))
    return out


def _mix(seed, T, a_set=(0, 1, 3, 16, 17, 33, 300), n_set=(0, 1, 64, 500), n_problems=14, metrics=None,
         thresholds=None, varied=False):
    return _far(_problems(seed, T, n_problems=n_problems, a_set=list(a_set), n_set=list(n_set), metrics=metrics,
                          thresholds=thresholds, varied=varied), seed)


def _engine(case):
    from frenetix_occlusion_b200.engine import MetricEngine
    return MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])


def _assert_host_equals_engine(probs, vehicles=None, want_pair=False, want_step=False, pinned=False, eng=None):
    eng = eng or _engine(probs[0][3])
    args = ([p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs])
    got = batch_host(eng, *args, vehicles=vehicles, want_pair=want_pair, want_step=want_step, pinned=pinned)
    want = engine_batch(eng, *args, vehicles=vehicles, want_pair=want_pair, want_step=want_step)
    _assert_same(got, want)
    return got


# ---------------------------------------------------------------------------------------------------- CPU
def _host_call(L, problems, n_traj, T=31, origins=True, agents=True, params=True, ego=True, valid=True,
               raw_agents=None, raw_stride=31, null_arrays=False, **common):
    """fo_metric_batch_host on descriptors (traj_begin, n_traj, n_agents, t_stride, table_offset) with host buffers that
    are never read: every case here must be rejected before the library touches them."""
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p)
    arr = (L.FoBatchProblem * max(len(problems), 1))()
    for i, (b, n, na, tp, off) in enumerate(problems):
        arr[i].traj_begin, arr[i].n_traj, arr[i].n_agents, arr[i].t_stride, arr[i].table_offset = b, n, na, tp, off
    raw = L.FoAgentsRaw()
    raw.n_agents = sum(q[2] for q in problems) if raw_agents is None else raw_agents
    raw.t_stride = raw_stride
    if not null_arrays:
        for f, _ in L.FoAgentsRaw._fields_[2:]:
            setattr(raw, f, p.value)
    n_problems = common.pop("n_problems", len(problems))
    a = L.FoMetricArgs()
    a.metric_mask = 0x7f
    for k, v in common.items():
        setattr(a, k, v)
    return L.lib.fo_metric_batch_host(p if ego else None, n_traj, T, p if origins else None,
                                      C.byref(raw) if agents else None, n_problems, arr, None,
                                      C.byref(a) if params else None, p if valid else None, p, p, None, None)


def test_batch_host_rejects_malformed_arguments_without_device():
    from frenetix_occlusion_b200 import _lib as L
    ok = [(0, 4, 2, 31, 0), (4, 3, 1, 31, 0)]
    # NULL arrays with problems
    for kw in ({"params": False}, {"ego": False}, {"origins": False}, {"agents": False}, {"valid": False},
               {"null_arrays": True}):
        assert _host_call(L, ok, 7, **kw) == FO_ERR_INVALID_ARG, kw
        assert b"fo_metric_batch_host" in L.lib.fo_last_error(), kw
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    raw, a = L.FoAgentsRaw(), L.FoMetricArgs()
    assert L.lib.fo_metric_batch_host(p, 4, 31, p, C.byref(raw), 1, None, None, C.byref(a), p, None, None, None,
                                      None) == FO_ERR_INVALID_ARG                                   # problems NULL
    # descriptors: the status fo_metric_batch gives the same rows (the library places the tables itself)
    for name, pr, n, T in (("gap", [(0, 4, 2, 31, 0), (5, 3, 2, 31, 0)], 8, 31),
                           ("order", [(4, 3, 2, 31, 0), (0, 4, 2, 31, 0)], 7, 31),
                           ("past n_traj", [(0, 4, 2, 31, 0), (4, 5, 2, 31, 0)], 8, 31),
                           ("uncovered", [(0, 4, 2, 31, 0)], 6, 31),
                           ("no states", [(0, 4, 2, 0, 0)], 4, 31),
                           ("negative", [(0, 4, -1, 31, 0)], 4, 31),
                           ("t_stride", [(0, 4, 2, 129, 0)], 4, 31),
                           ("T", [(0, 4, 2, 31, 0)], 4, 129),
                           ("T = 0", [(0, 4, 2, 31, 0)], 4, 0)):
        layout = np.array([[q[2], q[3]] for q in pr], dtype=np.int64)
        off = np.zeros(len(pr), dtype=np.int64)
        for i in range(1, len(pr)):
            off[i] = off[i - 1] + (L.lib.fo_agent_table_bytes(int(layout[i - 1, 0]), int(layout[i - 1, 1])) + 15) // 16 * 16
        dev = L.lib.fo_metric_batch(C.byref(_batch_args(L, [q[:4] + (int(o),) for q, o in zip(pr, off)], n, T)), None)
        got = _host_call(L, pr, n, T, raw_agents=max(sum(q[2] for q in pr), 0), raw_stride=129)
        assert dev < 0 and got == dev, (name, got, dev)
        assert b"fo_metric_batch_host" in L.lib.fo_last_error(), name
    assert _host_call(L, ok, 7, raw_agents=4) == FO_ERR_INVALID_ARG                                  # agents do not add up
    assert _host_call(L, [(0, 4, 2, 51, 0)], 4, raw_stride=31) == FO_ERR_INVALID_ARG                  # row stride too small
    assert b"t_stride 51 > raw row stride 31" in L.lib.fo_last_error()
    assert _host_call(L, ok, 7, n_peers=1) == FO_ERR_UNSUPPORTED
    assert _host_call(L, ok, 7, n_problems=-1) == FO_ERR_INVALID_ARG
    assert _host_call(L, ok, 7, metric_mask=1 << 4) == FO_ERR_INVALID_ARG                              # 'be' needs 'ttc'
    # nothing to do: no device work, so these pass on a machine without a GPU
    assert _host_call(L, [], 0) == 0
    assert _host_call(L, [(0, 0, 2, 31, 0), (0, 0, 0, 0, 0)], 0, ego=False, valid=False) == 0


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("outputs", ["summary", "pair", "step", "both"])
@pytest.mark.parametrize("fleet", [False, True])
def test_batch_host_equals_the_engine_batch(T, outputs, fleet, cuda_device):
    """Agent counts 0-300 (problems without agents among them) and trajectory counts 0-500 (problems without
    trajectories among them), every problem kilometres from the others at UTM-sized coordinates."""
    probs = _mix(T + 400 + 10 * fleet, T)
    assert {p[0].n_agents for p in probs} == {0, 1, 3, 16, 17, 33, 300} and {len(p[2]) for p in probs} == {0, 1, 64, 500}
    vehicles = _fleet(len(probs), T) if fleet else None
    _assert_host_equals_engine(probs, vehicles, outputs in ("pair", "both"), outputs in ("step", "both"))


@pytest.mark.gpu
def test_batch_host_equals_the_engine_batch_on_varied_agents(cuda_device):
    probs = _mix(451, 51, varied=True)
    _assert_host_equals_engine(probs, _fleet(len(probs), 51), True, True)


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", [None, "default", ["dce", "ttc", "wttc"], ["ttc", "be", "hr", "cp"]])
@pytest.mark.parametrize("armed", [False, True])
@pytest.mark.parametrize("detail", [False, True])
def test_batch_host_equals_the_engine_batch_metrics_and_thresholds(metrics, armed, detail, cuda_device):
    """Armed dce / ttc / be thresholds run the float64 rounding-tie variants."""
    from frenetix_occlusion_b200 import synthetic as S
    m = S.DEFAULT_METRICS if metrics == "default" else metrics
    thr = dict(S.DEFAULT_THRESHOLDS, dce=0.5, ttc=1.5, be=0.8) if armed else None
    probs = _mix(57 + armed, 31, metrics=m, thresholds=thr, n_set=(0, 1, 64, 200))
    _assert_host_equals_engine(probs, _fleet(len(probs), 57), detail, detail)


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_batch_host_takes_pageable_and_page_locked_inputs(pinned, cuda_device):
    probs = _mix(61, 51, a_set=(0, 5, 40), n_set=(300, 0, 700), n_problems=6)
    _assert_host_equals_engine(probs, _fleet(len(probs), 61), pinned=pinned)
    _assert_host_equals_engine(probs, None, True, True, pinned=pinned)


@pytest.mark.gpu
def test_batch_host_rounds_after_the_float64_shift(cuda_device):
    """At 4-6e6 m a float32 step is 0.25-0.5 m: rounding the world coordinates before the shift gives another bundle and
    other results, and the call gives those of the bundle rounded after the shift."""
    probs = _mix(67, 31, a_set=(6, 20), n_set=(200, 150), n_problems=2)
    origins = [(4.1e6 + 0.3, 5.3e6 + 0.7), (5.9e6 + 0.45, 4.4e6 + 0.15)]
    for i, (ag, origin, ego, case) in enumerate(probs):
        d = np.subtract(origins[i], origin)
        ego[..., 0] += d[0]
        ego[..., 1] += d[1]
        live = np.arange(ag.t_stride)[None, :] < ag.n_states[:, None]
        ag.x, ag.y = ag.x + d[0] * live, ag.y + d[1] * live
        probs[i] = (ag, origins[i], ego, case)
    eng = _engine(probs[0][3])
    ags, egos = [p[0] for p in probs], [p[2] for p in probs]
    after = [(e - np.array([o[0], o[1], 0, 0, 0])).astype(np.float32) for e, o in zip(egos, origins)]
    before = [e.astype(np.float32) - np.array([o[0], o[1], 0, 0, 0], dtype=np.float32) for e, o in zip(egos, origins)]
    differ = np.mean(np.concatenate([(a != b)[..., :2].ravel() for a, b in zip(after, before)]))
    assert differ > 0.5, differ
    got = _assert_host_equals_engine(probs, want_pair=True)
    zero = [(0.0, 0.0)] * len(probs)
    # agents stay in their own frames: the same float32 arrays with a zero origin
    shifted = [_shift_agents(ag, o) for ag, o in zip(ags, origins)]
    right = batch_host(eng, shifted, zero, [a.astype(np.float64) for a in after], want_pair=True)
    wrong = batch_host(eng, shifted, zero, [b.astype(np.float64) for b in before], want_pair=True)
    _assert_same(got, right)
    assert not np.array_equal(got["summary"], wrong["summary"], equal_nan=True)
    assert not np.array_equal(got["pair"], wrong["pair"], equal_nan=True)


def _shift_agents(ag, origin):
    """A copy of an AgentSet whose float64 positions are the float32 values fo_metric_batch_host gets for them."""
    import copy
    out = copy.copy(ag)
    out.x = (ag.x - origin[0]).astype(np.float32).astype(np.float64)
    out.y = (ag.y - origin[1]).astype(np.float32).astype(np.float64)
    return out


def chunked_run():
    """Run in a process of its own with FO_HOST_CHUNK_MB=1 (read once per process): a 12 MB float64 bundle crosses PCIe
    in several chunks, each with its own ingest launch.  Prints the chunk count the library's rule gives, the launches
    of the call beyond those of the engine path, and whether the outputs agree."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    probs = _mix(71, 51, a_set=(3, 0, 20), n_set=(1000,), n_problems=6)
    eng = _engine(probs[0][3])
    args = ([p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs])
    fleet = _fleet(len(probs), 71)
    n0 = L.lib.fo_launch_count()
    want = engine_batch(eng, *args, vehicles=fleet)
    torch.cuda.synchronize()
    n1 = L.lib.fo_launch_count()
    got = batch_host(eng, *args, vehicles=fleet)
    n2 = L.lib.fo_launch_count()
    N, row = sum(len(e) for e in args[2]), 51 * 5 * 8
    first = (1 << 20) // row + (1 if (1 << 20) % row else 0)
    bounds, at, step = [], 0, first
    while at < N:
        at = min(at + step, N)
        bounds.append(at)
        step *= 4
    equal = True
    try:
        _assert_same(got, want)
    except AssertionError:
        equal = False
    print(json.dumps({"chunks": len(bounds), "extra_launches": (n2 - n1) - (n1 - n0), "equal": equal}))


@pytest.mark.gpu
def test_batch_host_uploads_in_chunks(cuda_device):
    env = dict(os.environ, FO_HOST_CHUNK_MB="1")
    code = f"import sys; sys.path[:0] = [{HERE!r}, {ROOT!r}]; import test_metric_batch_host as M; M.chunked_run()"
    r = subprocess.run([sys.executable, "-s", "-c", code], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["chunks"] >= 3 and res["extra_launches"] == res["chunks"], res
    assert res["equal"], res


@pytest.mark.gpu
def test_batch_host_reuses_and_grows_its_workspace(cuda_device):
    small = _mix(73, 31, a_set=(2, 0), n_set=(10, 30), n_problems=2)
    large = _mix(79, 31, a_set=(0, 40, 300, 5), n_set=(500, 800, 64, 1000), n_problems=5)
    eng = _engine(small[0][3])
    _assert_host_equals_engine(small, eng=eng)
    _assert_host_equals_engine(large, want_pair=True, want_step=True, eng=eng)
    _assert_host_equals_engine(small, want_step=True, eng=eng)
    _assert_host_equals_engine(large, _fleet(len(large), 79), eng=eng)


@pytest.mark.gpu
def test_two_problems_of_a_host_batch_match_the_oracle(cuda_device):
    import parity
    from oracle import metric_oracle as MO
    from test_metric_gpu import _check
    probs = _mix(83, 31, a_set=(3, 17), n_set=(60, 25), n_problems=2)
    fleet = _fleet(2, 83)
    eng = _engine(probs[0][3])
    got = batch_host(eng, [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs], vehicles=fleet,
                     want_pair=True, want_step=True)
    row = q = 0
    for (ag, origin, ego, case), veh in zip(probs, fleet):
        n, a, T = len(ego), ag.n_agents, ego.shape[1]
        sub = dict(case, vehicle=dict(veh), ego=(ego - np.array([origin[0], origin[1], 0, 0, 0])).astype(np.float32)
                   .astype(np.float64), agents=[dict(x, pos=np.asarray(x["pos"])) for x in case["agents"]])
        # the oracle runs in the problem's own frame: the same float64 shift, then float32
        for x, k in zip(sub["agents"], range(a)):
            m = int(ag.n_states[k])
            x["pos"] = np.stack((ag.x[k, :m] - origin[0], ag.y[k, :m] - origin[1]), -1).astype(np.float32).astype(np.float64)
        out = MO.evaluate_bundle(sub)
        res = {"valid": got["valid"][row:row + n], "summary": got["summary"][row:row + n],
               "flags": got["flags"][row:row + n],
               "pair": got["pair"][q * 12:(q + n * a) * 12].reshape(n, a, 12),
               "step": got["step"][q * (T - 1) * 3:(q + n * a) * (T - 1) * 3].reshape(n, a, T - 1, 3)}
        _check(parity.compare_bundle(out, res, sub))
        row, q = row + n, q + n * a
