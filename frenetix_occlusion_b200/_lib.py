"""ctypes binding of ``libfo_b200.so`` (C ABI declared in ``include/fo_b200.h``).

There is no CPU fallback: if the shared library has not been built (``python __graft_entry__.py``
or ``make -C frenetix_occlusion_b200/csrc``) importing this module raises ``ImportError``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FO_LIB_PATH") or os.path.join(_HERE, "libfo_b200.so")   # FO_LIB_PATH: A/B builds

FO_OK = 0
FO_MAX_STATES = 128
FO_MAX_PEERS = 8
FO_SUMMARY_K = 10
FO_PAIR_K = 12
FO_STEP_K = 3
FO_VALID_SKIPPED = 2     # fo_metric_batch_select: a row ranked after its problem's first valid row, not assessed

# metric bits (FO_M_*), threshold bits (FO_T_*), kinds (FO_KIND_*), flags (FO_F_*)
M_BITS = {"cp": 1 << 0, "dce": 1 << 1, "ttc": 1 << 2, "hr": 1 << 3, "be": 1 << 4, "ttce": 1 << 5, "wttc": 1 << 6}
T_BITS = {"harm": 1 << 0, "risk": 1 << 1, "be": 1 << 2, "cp": 1 << 3, "ttc": 1 << 4, "dce": 1 << 5}
KINDS = {"pedestrian": 0, "bicycle": 1, "car": 2, "truck": 3, "bus": 4, "motorcycle": 5, "priorityvehicle": 6,
         "parkedvehicle": 7, "taxi": 8, "train": 9, "unknown": 10}
F_BE_RANGE = 1 << 0

SUMMARY_FIELDS = ("max_ego_risk_all", "max_obst_risk_all", "max_ego_harm_all", "max_obst_harm_all",
                  "max_collision_probability_all", "max_obst_harm_with_cp_all", "min_dce", "wttc",
                  "max_break_threat_number", "max_required_constant_deceleration")
PAIR_FIELDS = ("dce", "time_dce", "max_ego_risk", "max_obst_risk", "max_obst_risk_index", "max_obst_harm_with_cp",
               "max_ego_harm", "max_obst_harm", "max_collision_probability", "required_constant_deceleration",
               "break_threat_number", "argmax_cp_index")


class FoVehicle(C.Structure):
    _fields_ = [("length", C.c_float), ("width", C.c_float), ("mass", C.c_float), ("wb_rear_axle", C.c_float),
                ("a_max", C.c_float)]


class FoHarmCoeffs(C.Structure):
    _fields_ = [("rs_const", C.c_float), ("rs_speed", C.c_float), ("rs_side", C.c_float), ("rs_rear", C.c_float),
                ("ia_const", C.c_float), ("ia_speed", C.c_float), ("ped_const", C.c_float), ("ped_speed", C.c_float)]


class FoAgentsRaw(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("t_stride", C.c_int32),
                ("x", C.c_void_p), ("y", C.c_void_p), ("yaw", C.c_void_p), ("v", C.c_void_p),
                ("var_x", C.c_void_p), ("var_y", C.c_void_p), ("n_states", C.c_void_p), ("kind", C.c_void_p),
                ("length", C.c_void_p), ("width", C.c_void_p), ("buf_length", C.c_void_p), ("buf_width", C.c_void_p)]


class FoMetricArgs(C.Structure):
    _fields_ = [("ego", C.c_void_p), ("n_traj", C.c_int32), ("n_states", C.c_int32),
                ("agent_table", C.c_void_p), ("n_agents", C.c_int32), ("t_stride", C.c_int32),
                ("vehicle", FoVehicle), ("harm", FoHarmCoeffs), ("dt", C.c_double),
                ("metric_mask", C.c_uint32), ("threshold_mask", C.c_uint32),
                ("thr_harm", C.c_double), ("thr_risk", C.c_double), ("thr_be", C.c_double),
                ("thr_cp", C.c_double), ("thr_ttc", C.c_double), ("thr_dce", C.c_double),
                ("valid", C.c_void_p), ("summary", C.c_void_p), ("flags", C.c_void_p),
                ("pair", C.c_void_p), ("step", C.c_void_p),
                ("n_peers", C.c_int32), ("reserved_", C.c_int32), ("peer_delta", C.c_int64 * FO_MAX_PEERS)]


class FoBatchProblem(C.Structure):
    _fields_ = [("traj_begin", C.c_int64), ("n_traj", C.c_int32), ("n_agents", C.c_int32), ("t_stride", C.c_int32),
                ("reserved_", C.c_int32), ("table_offset", C.c_int64)]


class FoMetricBatchArgs(C.Structure):
    _fields_ = [("common", FoMetricArgs), ("n_problems", C.c_int32), ("reserved_", C.c_int32),
                ("problems", C.POINTER(FoBatchProblem)), ("arena_bytes", C.c_size_t)]


class FoPeerHandle(C.Structure):
    _fields_ = [("bytes", C.c_uint8 * 64)]


class FoVisibilityArgs(C.Structure):
    _fields_ = [("n_frames", C.c_int32), ("n_rays", C.c_int32), ("n_obstacles", C.c_int32), ("n_boundary", C.c_int32),
                ("ego", C.c_void_p), ("rect", C.c_void_p), ("rect_flags", C.c_void_p), ("boundary", C.c_void_p),
                ("sensor_radius", C.c_float), ("sensor_angle_deg", C.c_float),
                ("range", C.c_void_p), ("hit", C.c_void_p), ("visible", C.c_void_p)]


class FoPointQueryArgs(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("n_obstacles", C.c_int32), ("n_boundary", C.c_int32), ("n_polygons", C.c_int32),
                ("ego", C.c_void_p), ("points", C.c_void_p), ("rect", C.c_void_p), ("rect_flags", C.c_void_p),
                ("boundary", C.c_void_p), ("poly_xy", C.c_void_p), ("poly_off", C.c_void_p),
                ("sensor_radius", C.c_float), ("sensor_angle_deg", C.c_float), ("occluded_radius", C.c_float),
                ("focus_obstacle", C.c_int32), ("focus_margin", C.c_float),
                ("flags", C.c_void_p), ("blocker", C.c_void_p), ("lanelets", C.c_void_p)]


class FoRasterSpec(C.Structure):
    _fields_ = [("cx", C.c_double), ("cy", C.c_double), ("cs", C.c_double), ("sn", C.c_double),
                ("hx", C.c_double), ("hy", C.c_double), ("cell", C.c_double), ("org_x", C.c_double), ("org_y", C.c_double),
                ("nx", C.c_int32), ("ny", C.c_int32)]


class FoRegionPredicate(C.Structure):
    _fields_ = [("lanelet_mask", C.c_uint64), ("want_flags", C.c_uint32), ("reject_flags", C.c_uint32),
                ("disc_x", C.c_double), ("disc_y", C.c_double), ("disc_r", C.c_double)]


class FoRasterResult(C.Structure):
    _fields_ = [("sum_x", C.c_double), ("sum_y", C.c_double), ("count", C.c_int32), ("contains", C.c_int32),
                ("n_outline", C.c_int32), ("n_components", C.c_int32)]


class FoSpawnRegionArgs(C.Structure):
    _fields_ = [("frame", FoPointQueryArgs), ("raster", FoRasterSpec), ("pred", FoRegionPredicate),
                ("probe_x", C.c_double), ("probe_y", C.c_double),
                ("label", C.c_void_p), ("size", C.c_void_p), ("best", C.c_void_p), ("mask_dilated", C.c_void_p),
                ("result", C.c_void_p)]


class FoSpawnRectArgs(C.Structure):
    _fields_ = [("frame", FoPointQueryArgs), ("raster", FoRasterSpec), ("pred", FoRegionPredicate),
                ("centre_from", C.c_void_p), ("region_mask", C.c_void_p),
                ("region_ox", C.c_double), ("region_oy", C.c_double), ("region_cell", C.c_double),
                ("region_n", C.c_int32), ("outline_cap", C.c_int32),
                ("mask", C.c_void_p), ("outline", C.c_void_p), ("result", C.c_void_p)]


class FoHitsOnRoadArgs(C.Structure):
    _fields_ = [("n_rays", C.c_int32), ("n_obstacles", C.c_int32), ("n_polygons", C.c_int32),
                ("range", C.c_void_p), ("hit", C.c_void_p), ("ego", C.c_void_p), ("poly_xy", C.c_void_p), ("poly_off", C.c_void_p),
                ("ego_x", C.c_double), ("ego_y", C.c_double), ("angle0", C.c_double), ("dangle", C.c_double),
                ("org_x", C.c_double), ("org_y", C.c_double), ("on_road", C.c_void_p)]


class FoRolloutCvArgs(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("n_states", C.c_int32), ("t_stride", C.c_int32), ("dt", C.c_double),
                ("var0", C.c_double), ("var_factor", C.c_double),
                ("x0", C.c_void_p), ("y0", C.c_void_p), ("v", C.c_void_p), ("phi", C.c_void_p),
                ("x", C.c_void_p), ("y", C.c_void_p), ("yaw", C.c_void_p), ("vel", C.c_void_p),
                ("var_x", C.c_void_p), ("var_y", C.c_void_p)]


class FoRolloutPathArgs(C.Structure):
    _fields_ = [("n_jobs", C.c_int32), ("n_states", C.c_int32), ("t_stride", C.c_int32), ("dt", C.c_double),
                ("t1", C.c_double), ("var0", C.c_double), ("var_factor", C.c_double),
                ("path_xy", C.c_void_p), ("path_off", C.c_void_p),
                ("x0", C.c_void_p), ("y0", C.c_void_p), ("v0", C.c_void_p),
                ("x", C.c_void_p), ("y", C.c_void_p), ("yaw", C.c_void_p), ("vel", C.c_void_p),
                ("var_x", C.c_void_p), ("var_y", C.c_void_p), ("sample", C.c_void_p)]


HIT_NONE, HIT_BOUNDARY = -1, -2
RECT_EXISTS, RECT_TRANSPARENT = 1, 2
PT_IN_SENSOR, PT_ON_ROAD, PT_SHADOWED, PT_IN_OBSTACLE, PT_VISIBLE, PT_OCCLUDED, PT_FOCUS_SHADOW, PT_FOCUS_NEAR = 1, 2, 4, 8, 16, 32, 64, 128

# every symbol include/fo_b200.h declares: name -> (restype, argtypes)
_PROTOS = {
    "fo_agent_table_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "fo_agents_pack": (C.c_int, [C.POINTER(FoAgentsRaw), C.POINTER(FoVehicle), C.c_void_p, C.c_size_t, C.c_void_p]),
    "fo_metric_bundle": (C.c_int, [C.POINTER(FoMetricArgs), C.c_void_p]),
    "fo_metric_stats": (C.c_int, [C.POINTER(FoMetricArgs), C.c_void_p, C.c_void_p]),
    "fo_agent_table_bytes_corr": (C.c_size_t, [C.c_int32, C.c_int32]),
    "fo_agents_pack_corr": (C.c_int, [C.POINTER(FoAgentsRaw), C.c_void_p, C.POINTER(FoVehicle), C.c_void_p, C.c_size_t,
                                      C.c_void_p]),
    "fo_metric_bundle_corr": (C.c_int, [C.POINTER(FoMetricArgs), C.c_void_p]),
    "fo_metric_bundle_corr_peers": (C.c_int, [C.POINTER(FoMetricArgs), C.c_void_p]),
    "fo_metric_stats_corr": (C.c_int, [C.POINTER(FoMetricArgs), C.c_void_p, C.c_void_p]),
    "fo_metric_bundle_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(FoAgentsRaw),
                                        C.POINTER(FoMetricArgs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "fo_agent_batch_layout": (C.c_size_t, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fo_agents_pack_batch": (C.c_int, [C.POINTER(FoAgentsRaw), C.c_int32, C.POINTER(FoBatchProblem),
                                       C.POINTER(FoVehicle), C.c_void_p, C.c_size_t, C.c_void_p]),
    "fo_metric_batch": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.c_void_p]),
    "fo_metric_batch_detail": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.c_void_p]),
    "fo_agents_pack_batch_vehicles": (C.c_int, [C.POINTER(FoAgentsRaw), C.c_int32, C.POINTER(FoBatchProblem),
                                                C.POINTER(FoVehicle), C.c_void_p, C.c_size_t, C.c_void_p]),
    "fo_metric_batch_vehicles": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.POINTER(FoVehicle), C.c_void_p]),
    "fo_metric_batch_detail_vehicles": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.POINTER(FoVehicle), C.c_void_p]),
    "fo_agent_batch_layout_corr": (C.c_size_t, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fo_agents_pack_batch_corr": (C.c_int, [C.POINTER(FoAgentsRaw), C.c_void_p, C.c_int32, C.POINTER(FoBatchProblem),
                                            C.c_void_p, C.POINTER(FoVehicle), C.c_void_p, C.c_size_t, C.c_void_p]),
    "fo_metric_batch_corr": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.c_void_p, C.POINTER(FoVehicle), C.c_void_p]),
    "fo_metric_batch_detail_corr": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.c_void_p, C.POINTER(FoVehicle),
                                              C.c_void_p]),
    "fo_metric_batch_select": (C.c_int, [C.POINTER(FoMetricBatchArgs), C.c_void_p, C.POINTER(FoVehicle), C.c_void_p,
                                         C.c_void_p]),
    "fo_metric_batch_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(FoAgentsRaw), C.c_int32,
                                       C.POINTER(FoBatchProblem), C.POINTER(FoVehicle), C.POINTER(FoMetricArgs),
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fo_metric_batch_host_corr": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(FoAgentsRaw),
                                            C.c_void_p, C.c_int32, C.POINTER(FoBatchProblem), C.c_void_p,
                                            C.POINTER(FoVehicle), C.POINTER(FoMetricArgs), C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "fo_visibility_raycast": (C.c_int, [C.POINTER(FoVisibilityArgs), C.c_void_p]),
    "fo_visibility_stats": (C.c_int, [C.POINTER(FoVisibilityArgs), C.c_void_p, C.c_void_p]),
    "fo_visibility_points": (C.c_int, [C.POINTER(FoPointQueryArgs), C.c_void_p]),
    "fo_visibility_hits_on_road": (C.c_int, [C.POINTER(FoHitsOnRoadArgs), C.c_void_p]),
    "fo_spawn_region": (C.c_int, [C.POINTER(FoSpawnRegionArgs), C.c_void_p]),
    "fo_spawn_rect": (C.c_int, [C.POINTER(FoSpawnRectArgs), C.c_void_p]),
    "fo_rollout_cv": (C.c_int, [C.POINTER(FoRolloutCvArgs), C.c_void_p]),
    "fo_rollout_path": (C.c_int, [C.POINTER(FoRolloutPathArgs), C.c_void_p]),
    "fo_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(FoPeerHandle)]),
    "fo_peer_open": (C.c_int, [C.POINTER(FoPeerHandle), C.POINTER(C.c_void_p)]),
    "fo_peer_close": (C.c_int, [C.c_void_p]),
    "fo_peer_free": (C.c_int, [C.c_void_p]),
    "fo_probe_fp32_peak": (C.c_int, [C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_void_p]),
    "fo_launch_count": (C.c_uint64, []),
    "fo_version": (C.c_int, []),
    "fo_last_error": (C.c_char_p, []),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)


class FoError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built -- run `python __graft_entry__.py` (or make -C "
                          "frenetix_occlusion_b200/csrc); this package has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)        # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc: int, what: str = ""):
    if rc != FO_OK:
        msg = lib.fo_last_error().decode("utf-8", "replace")
        raise FoError(f"{what or 'libfo_b200'} failed with status {rc}: {msg}")
