"""The first valid row of every problem from host memory (fo_metric_batch_host_select): the inputs of
fo_metric_batch_host_corr, rank windows assessed in rounds, only the rows of those windows copied to the device.

CPU: declaration and export, every argument check without a device, the code-size budget of the window ingest kernel.
GPU (-m gpu): selected equals the first valid row of fo_metric_batch_host_corr on the same arguments and every row that is
assessed equals that call's row bit for bit, while skipped rows keep their sentinel summary / flags; first valid rows at
the window boundaries; page-locked and pageable inputs give the same bytes; the device path (MetricEngine.select_batch)
gives the same selection; a fleet whose first rows are valid assesses no more than the first window of each problem."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from kernel_sizes import size_of
from test_metric_batch_host import _mix, _params, _pinned, _raw_host
from test_metric_batch_host_corr import _corr_mix, _correlate, _cov_host, _cpu_batch, _cpu_params, _engine
from test_metric_batch_vehicles import _fleet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FO_ERR_INVALID_ARG, FO_ERR_UNSUPPORTED = -1, -2
SKIPPED = 2
ARMED = {"harm": 0.1, "risk": 0.01, "be": 1.0, "cp": 0.05, "ttc": 2.0, "wttc": None, "ttce": None, "dce": 2.0}
SUM_FILL, FLAG_FILL = -3.0, 0xDEADBEEF


def _inputs(L, agent_sets, origins, egos, vehicles=None, corr=None, pinned=False):
    """Host buffers of a batch as both host calls take them.  corr: the flags (default: the sets with cov_xy); "null"
    passes corr_host = NULL."""
    from frenetix_occlusion_b200.engine import vehicle_struct
    P = len(agent_sets)
    alloc = (lambda shape, dtype: _pinned(shape, dtype)) if pinned else np.zeros
    org = alloc((P, 2), np.float64)
    org[:] = np.asarray(origins, dtype=np.float64).reshape(P, 2)
    raw, n_agents, t_stride = _raw_host(L, agent_sets, org, alloc)
    cov = _cov_host(agent_sets, n_agents, t_stride, alloc)
    flags = None if corr == "null" else \
        np.array([a.cov_xy is not None for a in agent_sets] if corr is None else corr, dtype=np.uint8)
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
    return dict(ego=ego, N=N, T=T, org=org, raw=raw, cov=cov, P=P, problems=problems, flags=flags, veh=veh,
                offsets=offsets)


def _flags_ptr(x):
    return x["flags"].ctypes.data if x["flags"] is not None else None


def _select(L, params, x, cov_null=False, summary=True, flags=True):
    """fo_metric_batch_host_select on _inputs, outputs prefilled with sentinels.  Returns the status and the outputs."""
    out = {"selected": np.full(max(x["P"], 1), -9, np.int32), "valid": np.full(x["N"], 7, np.uint8)}
    if summary:
        out["summary"] = np.full((x["N"], L.FO_SUMMARY_K), SUM_FILL, np.float32)
    if flags:
        out["flags"] = np.full(x["N"], FLAG_FILL, np.uint32)
    ptr = lambda k: out[k].ctypes.data if k in out else None  # noqa: E731
    rc = L.lib.fo_metric_batch_host_select(x["ego"].ctypes.data, x["N"], x["T"], x["org"].ctypes.data, C.byref(x["raw"]),
                                           None if cov_null else x["cov"].ctypes.data, x["P"], x["problems"],
                                           _flags_ptr(x), x["veh"], C.byref(params), ptr("selected"), ptr("valid"),
                                           ptr("summary"), ptr("flags"))
    out["selected"] = out["selected"][:x["P"]]
    return rc, out


def _full(L, params, x):
    """fo_metric_batch_host_corr on the same inputs (all-zero flags for a NULL corr_host)."""
    out = {"valid": np.empty(x["N"], np.uint8), "summary": np.empty((x["N"], L.FO_SUMMARY_K), np.float32),
           "flags": np.empty(x["N"], np.uint32)}
    flags = x["flags"] if x["flags"] is not None else np.zeros(max(x["P"], 1), np.uint8)
    L.check(L.lib.fo_metric_batch_host_corr(x["ego"].ctypes.data, x["N"], x["T"], x["org"].ctypes.data,
                                            C.byref(x["raw"]), x["cov"].ctypes.data, x["P"], x["problems"],
                                            flags.ctypes.data, x["veh"], C.byref(params), out["valid"].ctypes.data,
                                            out["summary"].ctypes.data, out["flags"].ctypes.data, None, None),
            "fo_metric_batch_host_corr")
    return out


def _assert_matches_full(got, full, offsets):
    """selected against the first valid row of the full call; assessed rows bit for bit; skipped rows untouched."""
    gv, fv = got["valid"], full["valid"]
    assert set(np.unique(gv)) <= {0, 1, SKIPPED}
    done = gv != SKIPPED
    assert np.array_equal(gv[done], fv[done])
    if "summary" in got:
        assert np.array_equal(got["summary"][done].view(np.int32), full["summary"][done].view(np.int32))
        assert np.all(got["summary"][~done] == SUM_FILL)
    if "flags" in got:
        assert np.array_equal(got["flags"][done], full["flags"][done])
        assert np.all(got["flags"][~done] == FLAG_FILL)
    for p in range(len(offsets) - 1):
        lo, hi = int(offsets[p]), int(offsets[p + 1])
        ok = np.flatnonzero(fv[lo:hi] == 1)
        want = int(ok[0]) if len(ok) else hi - lo
        assert got["selected"][p] == want, (p, got["selected"][p], want, hi - lo)
        assert np.all(done[lo:lo + min(want + 1, hi - lo)]), p         # every rank up to the selected one is assessed


def _head(got, offsets):
    """The outputs that do not depend on timing: selected, and every output of the ranks up to each selected one.  A
    row ranked after its problem's selected row, in the same window, is assessed or skipped depending on when the
    valid row was found."""
    rows = np.concatenate([np.arange(int(offsets[p]), int(offsets[p]) + min(int(s) + 1, int(offsets[p + 1] - offsets[p])))
                           for p, s in enumerate(got["selected"])] + [np.zeros(0, np.int64)])
    return [got["selected"].tobytes()] + [got[k][rows].tobytes() for k in ("valid", "summary", "flags") if k in got]


def _team_warps(n_traj, T, a_min, sms):
    """pick_team_warps (fo_metric_sweep.cu): the team size of the batch."""
    lg = next(lg for lg in range(6) if (1 << lg) >= a_min or lg == 5)
    return max(1, min(sms * 8 * 4 // max(n_traj, 1), T // (4 * (32 >> lg)), 8))


def _w0(n_traj, T, a_min, n_run):
    """The first window (DESIGN.md 5.15): at least one rank per resident team, at least 32."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    teams = sms * 8 * 4 // _team_warps(n_traj, T, a_min, sms)
    return max(32, -(-teams // n_run))


# ---------------------------------------------------------------------------------------------------- CPU
def test_host_select_is_declared_and_exported():
    from frenetix_occlusion_b200 import _lib as L
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fo_b200.h")).read(), flags=re.S)
    assert re.search(r"\bfo_metric_batch_host_select\s*\(", text)
    assert "fo_metric_batch_host_select" in L.EXPORTED_SYMBOLS and hasattr(L.lib, "fo_metric_batch_host_select")


def test_host_select_checks_its_arguments_without_device():
    from frenetix_occlusion_b200 import _lib as L
    f = L.lib.fo_metric_batch_host_select
    params = _cpu_params(L)
    ags, origins, egos = _cpu_batch()
    x = _inputs(L, ags, origins, egos)
    sel = np.zeros(4, np.int32)
    valid = np.zeros(x["N"], np.uint8)
    call = lambda selected=sel.ctypes.data, pa=params, cov=x["cov"].ctypes.data, fl=_flags_ptr(x): f(  # noqa: E731
        x["ego"].ctypes.data, x["N"], x["T"], x["org"].ctypes.data, C.byref(x["raw"]), cov, x["P"], x["problems"], fl,
        None, C.byref(pa), selected, valid.ctypes.data, None, None)
    # NULL out_selected with problems
    assert call(selected=None) == FO_ERR_INVALID_ARG
    assert b"fo_metric_batch_host_select: out_selected" in L.lib.fo_last_error()
    # NULL cov_xy with a flagged problem that has agents; not with a NULL corr_host
    assert call(cov=None) == FO_ERR_INVALID_ARG
    assert L.lib.fo_last_error().startswith(b"fo_metric_batch_host_select: cov_xy") and b"problem 2" in L.lib.fo_last_error()
    # peer stores
    peers = _cpu_params(L)
    peers.n_peers = 1
    assert call(pa=peers) == FO_ERR_UNSUPPORTED and b"fo_metric_batch_host_select" in L.lib.fo_last_error()
    # a covariance that is not positive definite, with fo_metric_batch_host_corr's message
    ag = ags[2]
    ag.cov_xy = ag.cov_xy.copy()
    ag.cov_xy[1, 7] = 1.0001 * np.sqrt(ag.var_x[1, 7] * ag.var_y[1, 7])
    bad = _inputs(L, ags, origins, egos)
    assert f(bad["ego"].ctypes.data, bad["N"], bad["T"], bad["org"].ctypes.data, C.byref(bad["raw"]),
             bad["cov"].ctypes.data, bad["P"], bad["problems"], _flags_ptr(bad), None, C.byref(params), sel.ctypes.data,
             valid.ctypes.data, None, None) == FO_ERR_INVALID_ARG
    assert L.lib.fo_last_error() == (b"fo_metric_batch_host_select: problem 2, agent 1: covariance 7 is not positive "
                                     b"definite")
    # malformed descriptors: fo_metric_batch_host_corr's status, this call's name
    for name, change in (("gap", lambda pr: setattr(pr[1], "traj_begin", pr[1].traj_begin + 1)),
                         ("t_stride", lambda pr: setattr(pr[0], "t_stride", 129)),
                         ("agents", lambda pr: setattr(pr[0], "n_agents", -1))):
        y = _inputs(L, ags, origins, egos)
        change(y["problems"])
        old = L.lib.fo_metric_batch_host_corr(y["ego"].ctypes.data, y["N"], y["T"], y["org"].ctypes.data,
                                              C.byref(y["raw"]), y["cov"].ctypes.data, y["P"], y["problems"],
                                              _flags_ptr(y), None, C.byref(params), valid.ctypes.data, None, None, None,
                                              None)
        new = f(y["ego"].ctypes.data, y["N"], y["T"], y["org"].ctypes.data, C.byref(y["raw"]), y["cov"].ctypes.data,
                y["P"], y["problems"], _flags_ptr(y), None, C.byref(params), sel.ctypes.data, valid.ctypes.data, None,
                None)
        assert old < 0 and new == old, (name, old, new)
        assert b"fo_metric_batch_host_select" in L.lib.fo_last_error(), name
    # no rows: every selection is 0 without a device; no problems: nothing is read
    empty = _inputs(L, _cpu_batch()[0], origins, [e[:0] for e in egos], corr="null")
    sel[:] = -1
    assert f(None, 0, empty["T"], empty["org"].ctypes.data, C.byref(empty["raw"]), None, empty["P"], empty["problems"],
             None, None, C.byref(params), sel.ctypes.data, None, None, None) == 0
    assert list(sel[:3]) == [0, 0, 0]
    assert f(None, 0, 31, None, None, None, 0, None, None, None, C.byref(params), None, None, None, None) == 0


def test_window_ingest_kernel_stays_inside_its_code_size_budget():
    """fo_ego_window_ingest_kernel: 2944 bytes when it was added (DESIGN.md 5.15) + 1 kB."""
    assert size_of("fo_ego_window_ingest_kernel") <= 2944 + 1024


# ---------------------------------------------------------------------------------------------------- GPU
def _check_mix(probs, vehicles=None, corr=None, eng=None, pinned=False, summary=True, flags=True):
    from frenetix_occlusion_b200 import _lib as L
    eng = eng or _engine(probs[0][3])
    params = _params(eng)
    x = _inputs(L, [p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs], vehicles, corr, pinned)
    rc, got = _select(L, params, x, summary=summary, flags=flags)
    L.check(rc, "fo_metric_batch_host_select")
    _assert_matches_full(got, _full(L, params, x), x["offsets"])
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("T", [31, 51])
@pytest.mark.parametrize("every, fleet", [(0, False), (1, True), (2, True), (2, False)],
                         ids=["diagonal-shared", "correlated-per-problem", "mixed-per-problem", "mixed-shared"])
def test_host_select_equals_the_first_valid_row_of_the_host_call(T, every, fleet, cuda_device, monkeypatch):
    """Agent counts 0, 1, 16, 17 and 40 (both sides of the window-filter / team class), N_p 0 to 1500, armed thresholds
    so rows fail, in batches of 1, 3, 17 and 256 problems at UTM-sized coordinates."""
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    for P in (1, 3, 17, 256):
        which = {0: "none", 1: "all", 2: "half"}[every]
        probs = _corr_mix(T * 11 + P + every, T, which, a_set=(0, 1, 16, 17, 40), n_set=(0, 1, 31, 200, 1500),
                          n_problems=P, thresholds=ARMED)
        _check_mix(probs, _fleet(P, T + P) if fleet else None)


@pytest.mark.gpu
@pytest.mark.parametrize("metrics", ["default", "all"])
@pytest.mark.parametrize("armed", [False, True], ids=["null", "armed"])
def test_host_select_with_metric_sets_and_thresholds(metrics, armed, cuda_device, monkeypatch):
    from frenetix_occlusion_b200 import synthetic as S
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    m = S.DEFAULT_METRICS if metrics == "default" else S.ALL_METRICS
    probs = _corr_mix(151 + armed, 31, "half", metrics=m, thresholds=ARMED if armed else None,
                      a_set=(0, 3, 17, 33), n_set=(0, 64, 700), n_problems=40)
    _check_mix(probs, _fleet(40, 151))


@pytest.mark.gpu
def test_host_select_without_flags_summary_or_flags(cuda_device, monkeypatch):
    """corr_host NULL (no problem correlated, cov_xy never read), and NULL out_summary / out_flags."""
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    probs = _mix(157, 31, a_set=(0, 5, 17, 40), n_set=(0, 100, 900), n_problems=20, thresholds=ARMED)
    offsets = np.concatenate([[0], np.cumsum([len(p[2]) for p in probs])])
    a = _check_mix(probs, corr="null")
    b = _check_mix(probs, corr="null", summary=False, flags=False)
    assert _head(a, offsets)[:2] == _head(b, offsets)


@pytest.mark.gpu
def test_host_select_under_a_forced_team_size(cuda_device, monkeypatch):
    """FO_TEAM_WARPS applies to the whole batch, as in fo_metric_batch_host_corr."""
    for warps in ("1", "4"):
        monkeypatch.setenv("FO_TEAM_WARPS", warps)
        probs = _corr_mix(163, 31, "half", a_set=(1, 17, 40), n_set=(64, 1000), n_problems=30, thresholds=ARMED)
        _check_mix(probs, _fleet(30, 163))


def _ranked_fleet(P, seed, corr):
    """P copies of one 1000-row problem (24 agents, armed thresholds) at a UTM-sized place; and the good / bad ranks of
    its rows from one full pass of fo_metric_batch_host_corr over that batch (the batch's own team size)."""
    from frenetix_occlusion_b200 import _lib as L
    from frenetix_occlusion_b200 import synthetic as S
    from frenetix_occlusion_b200.engine import AgentSet
    from test_metric_batch_host import _far
    case = S.make_case(1000, 24, 31, seed=seed, thresholds=ARMED)
    prob = _far([(AgentSet.from_case(case["agents"]), (0.0, 0.0), case["ego"], case)], seed)[0]
    if corr:
        prob = _correlate(prob, seed)
    ag, origin, ego, case = prob
    eng = _engine(case)
    x = _inputs(L, [ag] * P, [origin] * P, [ego] * P)
    valid = _full(L, _params(eng), x)["valid"][:1000]
    good, bad = np.flatnonzero(valid == 1), np.flatnonzero(valid == 0)
    assert len(good) >= 1 and len(bad) >= 1, (len(good), len(bad))
    return eng, ag, origin, ego, good, bad


@pytest.mark.gpu
@pytest.mark.parametrize("corr", [False, True], ids=["diagonal", "correlated"])
def test_first_valid_row_at_the_window_boundaries(corr, cuda_device, monkeypatch):
    """256 problems of 1000 rows reordered so that the first valid row sits at rank 0, w0 - 1, w0, w0 + 1, at the ends
    and starts of the next windows, at the last row, or nowhere; rows are repeated to fill the bundle."""
    from frenetix_occlusion_b200 import _lib as L
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    P, N = 256, 1000
    eng, ag, origin, ego, good, bad = _ranked_fleet(P, 5 + corr, corr)
    w0 = _w0(P * N, 31, 24, P)
    ranks = [0, w0 - 1, w0, w0 + 1, 5 * w0 - 1, 5 * w0, 5 * w0 + 1, 21 * w0 - 1, 21 * w0, N - 1, None]
    assert 21 * w0 < N
    egos, want = [], []
    for p in range(P):
        r = ranks[p % len(ranks)]
        order = np.resize(bad, N)
        if r is not None:
            order[r] = good[p % len(good)]
        egos.append(ego[order])
        want.append(N if r is None else r)
    x = _inputs(L, [ag] * P, [origin] * P, egos)
    rc, got = _select(L, _params(eng), x)
    L.check(rc, "fo_metric_batch_host_select")
    assert list(got["selected"]) == want
    _assert_matches_full(got, _full(L, _params(eng), x), x["offsets"])


@pytest.mark.gpu
def test_page_locked_and_pageable_rows_give_the_same_bytes(cuda_device, monkeypatch):
    """Both staging routes: rows read in place (torch pin_memory) and rows copied window by window (numpy).  Each
    equals fo_metric_batch_host_corr wherever it assessed a row; selected and the ranks up to it are byte-identical."""
    from frenetix_occlusion_b200 import _lib as L
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    probs = _corr_mix(167, 51, "half", a_set=(0, 5, 17, 40), n_set=(0, 300, 1200), n_problems=24, thresholds=ARMED)
    eng = _engine(probs[0][3])
    args = ([p[0] for p in probs], [p[1] for p in probs], [p[2] for p in probs], _fleet(24, 167))
    outs = []
    for pinned in (False, True):
        x = _inputs(L, *args, pinned=pinned)
        rc, got = _select(L, _params(eng), x)
        L.check(rc, "fo_metric_batch_host_select")
        _assert_matches_full(got, _full(L, _params(eng), x), x["offsets"])
        outs.append(got)
    assert _head(outs[0], x["offsets"]) == _head(outs[1], x["offsets"])


@pytest.mark.gpu
@pytest.mark.parametrize("every", [0, 2], ids=["diagonal", "mixed"])
def test_host_select_equals_the_device_select(every, cuda_device, monkeypatch):
    """MetricEngine.set_agent_batch + select_batch on the same fleet picks the same rows."""
    import torch
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    which = {0: "none", 2: "half"}[every]
    probs = _corr_mix(173 + every, 31, which, a_set=(0, 1, 17, 40), n_set=(0, 1, 64, 1000), n_problems=33,
                      thresholds=ARMED)
    fleet = _fleet(33, 173)
    got = _check_mix(probs, fleet)
    eng = _engine(probs[0][3])
    eng.set_agent_batch([p[0] for p in probs], [p[1] for p in probs], vehicles=fleet, correlated=True)
    r = eng.select_batch([p[2] for p in probs])
    torch.cuda.synchronize()
    assert np.array_equal(r.selected.cpu().numpy(), got["selected"])


@pytest.mark.gpu
def test_early_exit_assesses_no_more_than_the_first_window(cuda_device, monkeypatch):
    """256 x 1000 x 31 with a valid row at rank 0 of every problem: one round, at most w0 rows assessed per problem."""
    from frenetix_occlusion_b200 import _lib as L
    monkeypatch.delenv("FO_TEAM_WARPS", raising=False)
    P, N = 256, 1000
    eng, ag, origin, ego, good, bad = _ranked_fleet(P, 5, False)
    order = np.concatenate([good[:1], np.resize(bad, N - 1)])
    for pinned in (False, True):
        x = _inputs(L, [ag] * P, [origin] * P, [ego[order]] * P, pinned=pinned)
        rc, got = _select(L, _params(eng), x)
        L.check(rc, "fo_metric_batch_host_select")
        assert np.all(got["selected"] == 0)
        w0 = _w0(P * N, 31, 24, P)
        assessed = (got["valid"] != SKIPPED).reshape(P, N).sum(axis=1)
        assert assessed.max() <= w0, (assessed.max(), w0)
        assert np.all(got["valid"].reshape(P, N)[:, w0:] == SKIPPED)
        _assert_matches_full(got, _full(L, _params(eng), x), x["offsets"])
