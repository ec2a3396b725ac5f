"""Per-pair and per-step detail for batches of independent planning problems (fo_metric_batch_detail,
MetricEngine.assess_batch(want_pair, want_step), batch.assess_interfaces(want_pair, want_step),
batch.prefetch_interfaces).  The CPU part checks the argument validation (before any CUDA call) and the code size of the
batched detail kernel; the GPU part checks that every problem of a batch gets exactly what the single-problem detail path
gives it, and that a prefetch over many interfaces serves the per-trajectory protocol as each interface's own would."""
import ctypes as C
import os
import re
import shutil
import subprocess
import types

import numpy as np
import pytest

from test_metric_batch import A_SET, N_SET, _batch_args, _engine, _problems, _scene_interface

FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2
SCENES = ("scene_scenario1.json", "scene_scenario2.json", "scene_scenario3.json", "scene_parked_car.json")


# ---------------------------------------------------------------------------------------------------- CPU
def test_batch_detail_argument_validation_without_device():
    from frenetix_occlusion_b200 import _lib as L
    run = lambda a: L.lib.fo_metric_batch_detail(C.byref(a), None)  # noqa: E731

    def args(problems, n_traj, T=31, pair=1 << 24, step=None):
        a = _batch_args(L, problems, n_traj, T)
        a.common.agent_table = 1 << 20             # never dereferenced by the host-side checks
        a.common.pair, a.common.step = pair, step
        return a
    assert L.lib.fo_metric_batch_detail(None, None) == FO_ERR_INVALID_ARG
    ok = [(0, 4, 2, 31, 0)]
    assert run(args(ok, 4, pair=None)) == FO_ERR_INVALID_ARG                                         # no detail buffer
    assert b"fo_metric_batch_detail" in L.lib.fo_last_error()
    assert run(args(ok, 4, pair=(1 << 24) + 8)) == FO_ERR_INVALID_ARG                                # misaligned pair
    assert run(args(ok, 4, pair=None, step=(1 << 24) + 2)) == FO_ERR_INVALID_ARG                     # misaligned step
    a = args(ok, 4)
    a.common.n_peers = 1
    assert run(a) == FO_ERR_UNSUPPORTED                                                              # peer stores
    a = args([], 0)
    a.n_problems = -1
    assert run(a) == FO_ERR_INVALID_ARG
    a = args(ok, 4)
    a.problems = None
    assert run(a) == FO_ERR_INVALID_ARG
    for step in (None, 1 << 26):                   # pair only, and pair + step
        assert run(args([(0, 4, 2, 31, 0), (5, 3, 2, 31, 4096)], 8, step=step)) == FO_ERR_INVALID_ARG  # gap between rows
        assert run(args([(4, 3, 2, 31, 0), (0, 4, 2, 31, 4096)], 7, step=step)) == FO_ERR_INVALID_ARG  # not in row order
        assert run(args([(0, 4, 2, 31, 0), (4, 5, 2, 31, 4096)], 8, step=step)) == FO_ERR_INVALID_ARG  # rows past n_traj
        assert run(args(ok, 6, step=step)) == FO_ERR_INVALID_ARG                                       # rows left uncovered
        assert run(args([(0, 4, 2, 31, (1 << 20) - 64)], 4, step=step)) == FO_ERR_INVALID_ARG         # table past the arena
        assert run(args([(0, 4, 2, 31, 8)], 4, step=step)) == FO_ERR_INVALID_ARG                       # misaligned table
        assert run(args([(0, 4, 2, 0, 0)], 4, step=step)) == FO_ERR_INVALID_ARG                        # agents, no states
        assert run(args([(0, 4, 2, 129, 0)], 4, step=step)) == FO_ERR_UNSUPPORTED                      # t_stride > FO_MAX_STATES
        assert run(args(ok, 4, T=129, step=step)) == FO_ERR_UNSUPPORTED                                # T > FO_MAX_STATES
    a = args(ok, 4)
    a.common.agent_table = (1 << 20) + 8
    assert run(a) == FO_ERR_INVALID_ARG                                                              # misaligned arena
    a = args(ok, 4)
    a.common.metric_mask = L.M_BITS["be"]
    assert run(a) == FO_ERR_INVALID_ARG                                                              # 'be' without 'ttc'
    a = args(ok, 4)
    a.common.valid = None
    assert run(a) == FO_ERR_INVALID_ARG
    a = args(ok, 4)
    a.common.summary = (1 << 24) + 4
    assert run(a) == FO_ERR_INVALID_ARG                                                              # misaligned summary
    assert b"fo_metric_batch_detail" in L.lib.fo_last_error()
    assert run(args([(0, 0, 0, 0, 0)], 0)) == 0                                                      # nothing to do


def test_batched_detail_kernel_stays_inside_the_instruction_cache_budget():
    """The batched detail kernel shares the detail kernel's body: it is held to that kernel's budgets in test_capi.py."""
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
    cold = {}
    elf = subprocess.run([cuobjdump, "-elf", L.LIB_PATH], capture_output=True, text=True).stdout
    for line in elf.splitlines():
        m = re.match(r"\s*0x[0-9a-f]+\s+0x[0-9a-f]+\s+(0x[0-9a-f]+)\s+.*\$(_ZN\S+?)\$(_ZN\S+)", line)
        if m and ("obb_round_mm_f64" in m.group(3) or "sincos_f64_of_f32" in m.group(3)):
            cold[m.group(2)] = cold.get(m.group(2), 0) + int(m.group(1), 16)

    def size_of(*parts):
        hit = [v - cold.get(k, 0) for k, v in sizes.items() if all(p in k for p in parts)]
        assert len(hit) == 1, (parts, sorted(sizes))
        return hit[0]
    assert size_of("fo_metric_batch_detail_kernel", "ILj127E") <= 50 * 1024   # all 7 metrics, incl. BE helpers
    assert size_of("fo_metric_batch_detail_kernel", "ILj111E") <= 38 * 1024   # default metrics


# ---------------------------------------------------------------------------------------------------- GPU
def _assert_equal(g, w, what):
    g, w = g.cpu().numpy(), w.cpu().numpy()
    assert g.shape == w.shape, (what, g.shape, w.shape)
    assert np.array_equal(g, w, equal_nan=True), what
    if g.dtype.kind == "f":
        assert np.array_equal(np.isnan(g), np.isnan(w)), what


def _assert_detail_batch_equals_single(problems, want_pair, want_step):
    import torch
    eng = _engine(problems[0][3])
    eng.set_agent_batch([p[0] for p in problems], [p[1] for p in problems])
    parts = eng.assess_batch([p[2] for p in problems], want_pair=want_pair, want_step=want_step).split()
    single = _engine(problems[0][3])
    for i, ((ag, origin, ego, _), got) in enumerate(zip(problems, parts)):
        assert (got.pair is not None) == want_pair and (got.step is not None) == want_step
        if not len(ego):
            assert got.valid.numel() == 0
            continue
        single.set_agents(ag, origin=origin)
        want = single.assess(ego, want_pair=want_pair, want_step=want_step)
        torch.cuda.synchronize()
        for f in ("valid", "flags", "summary") + (("pair",) if want_pair else ()) + (("step",) if want_step else ()):
            _assert_equal(getattr(got, f), getattr(want, f), (i, f, ag.n_agents, len(ego)))


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 31, 51, 128])
@pytest.mark.parametrize("detail", ["pair", "step", "both"])
def test_detail_batch_equals_single_problem_path(T, detail, cuda_device):
    probs = _problems(T + 100, T)
    assert {p[0].n_agents for p in probs} == set(A_SET) and {len(p[2]) for p in probs} == set(N_SET)
    _assert_detail_batch_equals_single(probs, detail != "step", detail != "pair")


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", [None, "default", ["hr", "cp"], ["dce", "ttc", "wttc"]])
@pytest.mark.parametrize("armed", [False, True])
def test_detail_batch_equals_single_problem_path_metrics_and_thresholds(metrics, armed, cuda_device):
    from frenetix_occlusion_b200 import synthetic as S
    m = S.DEFAULT_METRICS if metrics == "default" else metrics
    thr = dict(S.DEFAULT_THRESHOLDS, dce=0.5, ttc=1.5, be=0.8) if armed else None
    _assert_detail_batch_equals_single(_problems(27 + armed, 31, metrics=m, thresholds=thr), True, True)


@pytest.mark.gpu
def test_every_problem_of_a_detail_batch_matches_the_oracle(cuda_device):
    _assert_every_detail_problem_matches_the_oracle(_problems(29, 31, a_set=[0, 3, 17, 40], n_set=[60, 25, 80, 30]))


@pytest.mark.gpu
def test_every_problem_of_a_detail_batch_matches_the_oracle_on_varied_agents(cuda_device):
    _assert_every_detail_problem_matches_the_oracle(_problems(30, 51, a_set=[0, 5, 17, 40], n_set=[60, 25, 80, 30],
                                                              varied=True))


def _assert_every_detail_problem_matches_the_oracle(probs):
    import parity
    from oracle import metric_oracle as MO
    from test_metric_gpu import _check
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs])
    parts = eng.assess_batch([p[2] for p in probs], want_pair=True, want_step=True).split()
    for (ag, origin, ego, case), got in zip(probs, parts):
        sub = dict(case, ego=ego - np.array([origin[0], origin[1], 0, 0, 0]),
                   agents=[dict(a, pos=np.asarray(a["pos"])) for a in case["agents"]])
        # the oracle runs in the problem's own frame: the same float64 shift the batch applies
        for a, k in zip(sub["agents"], range(ag.n_agents)):
            n = int(ag.n_states[k])
            a["pos"] = np.stack((ag.x[k, :n] - origin[0], ag.y[k, :n] - origin[1]), -1).astype(np.float32).astype(np.float64)
        sub["ego"] = sub["ego"].astype(np.float32).astype(np.float64)
        out = MO.evaluate_bundle(sub)
        res = {"valid": got.valid.cpu().numpy(), "summary": got.summary.cpu().numpy(),
               "flags": got.flags.cpu().numpy().astype(np.uint32), "pair": got.pair.cpu().numpy(),
               "step": got.step.cpu().numpy()}
        _check(parity.compare_bundle(out, res, sub))


@pytest.mark.gpu
def test_assess_interfaces_with_detail_equals_each_interface(cuda_device):
    import torch
    from frenetix_occlusion_b200.batch import assess_interfaces
    pairs = [_scene_interface(n) for n in SCENES]
    fos, fans = [p[0] for p in pairs], [p[1] for p in pairs]
    got = assess_interfaces(fos, fans, want_pair=True, want_step=True)
    for fo, fan, g in zip(fos, fans, got):
        want = fo.assess_bundle(fan, True, True)
        torch.cuda.synchronize()
        for f in ("valid", "flags", "summary", "pair", "step"):
            _assert_equal(getattr(g, f), getattr(want, f), f)


class _Cart:
    """trajectory.cartesian of the reference's planner: a fresh array per attribute access"""
    def __init__(self, arr):
        self._a = arr
    x = property(lambda self: np.array(self._a[:, 0]))
    y = property(lambda self: np.array(self._a[:, 1]))
    theta = property(lambda self: np.array(self._a[:, 2]))
    v = property(lambda self: np.array(self._a[:, 3]))
    a = property(lambda self: np.array(self._a[:, 4]))


def _trajectories(fan):
    return [types.SimpleNamespace(cartesian=_Cart(np.array(e, dtype=np.float64))) for e in fan]


def _assert_same_assessments(got, want):
    from oracle.compare import compare_results
    for (rg, okg), (rw, okw) in zip(got, want):
        assert okg == okw
        assert not compare_results(rw, rg, rtol=0, atol=0) and not compare_results(rg, rw, rtol=0, atol=0)


@pytest.mark.gpu
def test_prefetch_interfaces_serves_every_candidate_like_each_interface(cuda_device):
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200.batch import prefetch_interfaces
    pairs = [_scene_interface(n) for n in SCENES]
    fos = [p[0] for p in pairs]
    cands = [_trajectories(p[1]) for p in pairs]
    idle, idle_fan = _scene_interface(SCENES[1])
    idle.agent_manager.reset()                          # an interface without phantom agents
    l0 = L.lib.fo_launch_count()
    counts = prefetch_interfaces(fos + [idle], cands + [_trajectories(idle_fan)])
    assert L.lib.fo_launch_count() - l0 == 3            # two pack launches and one detail launch for all interfaces
    assert counts == [len(c) for c in cands] + [0]
    l0 = L.lib.fo_launch_count()
    served = [[fo.trajectory_safety_assessment(t) for t in c] for fo, c in zip(fos, cands)]
    assert L.lib.fo_launch_count() == l0, "prefetched trajectories must not launch again"
    assert idle.trajectory_safety_assessment(_trajectories(idle_fan)[0]) == ({}, True)
    # a trajectory outside the candidate list packs the interface's table and gets the single-path result
    extra = []
    for fo, c in zip(fos, cands):
        arr = np.array(c[0].cartesian._a)
        arr[:, 3] += 0.25
        t = types.SimpleNamespace(cartesian=_Cart(arr))
        extra.append((t, fo.trajectory_safety_assessment(t)))
    for fo, c, s, (t, x) in zip(fos, cands, served, extra):
        core = fo.metrics._core
        core._fingerprint = None                        # the interface's own path from scratch: sync, pack, prefetch
        assert fo.prefetch_assessments(c) == len(c)
        own = [fo.trajectory_safety_assessment(t) for t in c]
        _assert_same_assessments(s, own)
        core._fingerprint = None
        _assert_same_assessments([x], [fo.trajectory_safety_assessment(t)])


@pytest.mark.gpu
def test_prefetch_interfaces_rejects_configurations_one_batch_cannot_share(cuda_device):
    from frenetix_occlusion_b200.batch import prefetch_interfaces
    pairs = [_scene_interface(n) for n in SCENES[:2]]
    fos, cands = [p[0] for p in pairs], [_trajectories(p[1]) for p in pairs]
    fos[1].metrics._core.engine.dt = fos[1].metrics._core.engine.dt * 2
    with pytest.raises(ValueError):
        prefetch_interfaces(fos, cands)
    fos[1].metrics._core.engine.dt = fos[0].metrics._core.engine.dt
    short = [types.SimpleNamespace(cartesian=_Cart(np.array(t.cartesian._a[:20]))) for t in cands[1]]
    with pytest.raises(ValueError):
        prefetch_interfaces(fos, [cands[0], short])
    with pytest.raises(ValueError):
        prefetch_interfaces(fos, cands[:1])
