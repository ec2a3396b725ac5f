"""The C-ABI library loads on a machine without a GPU and exports every symbol the header declares;
argument validation works without touching the device."""
import ctypes as C
import os
import re

from conftest import ROOT
from kernel_sizes import size_of


def _header_functions():
    text = open(os.path.join(ROOT, "include", "fo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fo_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported():
    from frenetix_occlusion_b200 import _lib as L
    names = _header_functions()
    assert len(names) >= 9
    raw = C.CDLL(L.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} declared in include/fo_b200.h but not exported by libfo_b200.so"
    assert set(names) == set(L.EXPORTED_SYMBOLS), set(names) ^ set(L.EXPORTED_SYMBOLS)


def test_argument_validation_without_device():
    from frenetix_occlusion_b200 import _lib as L
    assert L.lib.fo_version() == 1
    assert L.lib.fo_agent_table_bytes(256, 51) == 256 * 51 * 40 + 256 * 32 + 256 * 51 * 24 + 256 * 7 * 20 + 256 * 8   # time-major copies, 7 windows of 8 steps, slot maps
    assert L.lib.fo_agent_table_bytes(33, 31) == 33 * 31 * 40 + 33 * 32 + 64 * 31 * 24 + 64 * 4 * 20 + 64 * 8
    assert L.lib.fo_metric_bundle(None, None) == -1
    assert b"NULL" in L.lib.fo_last_error()
    a = L.FoMetricArgs()
    a.n_traj = -3
    assert L.lib.fo_metric_bundle(C.byref(a), None) == -1
    a.n_traj, a.n_states = 4, 4000          # T beyond FO_MAX_STATES, pointers non-NULL
    buf = (C.c_float * 16)()
    a.ego = C.cast(buf, C.c_void_p)
    a.valid = C.cast(buf, C.c_void_p)
    assert L.lib.fo_metric_bundle(C.byref(a), None) == -2
    v = L.FoVisibilityArgs()
    v.n_frames, v.n_rays = 1, 8
    assert L.lib.fo_visibility_raycast(C.byref(v), None) == -1      # NULL arrays
    r = L.FoRolloutCvArgs()
    r.n_agents, r.n_states, r.t_stride = 2, 31, 8
    assert L.lib.fo_rollout_cv(C.byref(r), None) == -1              # stride < states
    # peer-mapped buffers: argument checks come before any CUDA call
    ptr, h = C.c_void_p(), L.FoPeerHandle()
    assert L.lib.fo_peer_alloc(0, C.byref(ptr), C.byref(h)) == -1 and L.lib.fo_peer_alloc(64, None, C.byref(h)) == -1
    assert L.lib.fo_peer_open(None, C.byref(ptr)) == -1 and L.lib.fo_peer_open(C.byref(h), None) == -1
    assert L.lib.fo_peer_close(None) == 0 and L.lib.fo_peer_free(None) == 0
    assert C.sizeof(L.FoPeerHandle) == 64 and L.FoMetricArgs.peer_delta.size == 8 * L.FO_MAX_PEERS
    assert L.lib.fo_spawn_region(None, None) == -1 and L.lib.fo_spawn_rect(None, None) == -1
    assert L.lib.fo_visibility_hits_on_road(None, None) == -1


def test_engine_refuses_to_run_without_cuda():
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from frenetix_occlusion_b200.engine import MetricEngine
    from frenetix_occlusion_b200 import synthetic as S
    with pytest.raises(RuntimeError):
        MetricEngine(S.VEHICLE, 0.1, S.ALL_METRICS, S.DEFAULT_THRESHOLDS)


def test_hot_kernels_stay_inside_the_instruction_cache_budget():
    """The summary and detail kernels are instruction-issue-bound and sit next to the 32 kB L1.5 instruction cache:
    inlined duplicates showed up as stall_no_inst and cost 25 % (summary, 70 kB -> 47 kB) and 2.6x (detail, 111 kB ->
    59 kB) -- DESIGN.md section 6.  Guard the code size of the shapes the benchmark and the planner use."""
    # the throughput kernel sits at the edge of the instruction cache: +2-5 kB cost 5-8 % in every experiment (DESIGN.md 5.1)
    assert size_of("fo_metric_sweep_kernel", "ILj127ELb0ELb1ELb0E", hot=True) <= 44 * 1024   # all 7 metrics, one-warp window-filter shape
    assert size_of("fo_metric_sweep_kernel", "ILj127ELb0ELb1ELb1E", hot=True) <= 52 * 1024   # ... with the float64 tie path (armed dce / ttc / be)
    assert size_of("fo_metric_sweep_kernel", "ILj111ELb0ELb1ELb0E", hot=True) <= 34 * 1024   # default metrics (no BE)
    assert size_of("fo_metric_sweep_kernel", "ILj127ELb0ELb0ELb0E", hot=True) <= 56 * 1024   # team shape (latency path)
    assert size_of("fo_metric_detail_kernel", "ILj127E", hot=True) <= 50 * 1024            # detail kernel (lane = agent), all 7 metrics, incl. BE helpers
    assert size_of("fo_metric_detail_kernel", "ILj111E", hot=True) <= 38 * 1024            # default metrics
