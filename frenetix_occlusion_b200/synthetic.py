"""Seeded synthetic workloads for the assessment hot path (SURVEY.md §8(d), BASELINE.json configs).

These generate *inputs* only (trajectory bundles, phantom-agent tables, obstacle frames); they are
used by ``bench.py`` and the tests.  All values are rounded to float32 and returned as float64, so
the fp32 CUDA path and the float64 oracle consume bit-identical inputs.
"""
from __future__ import annotations

import numpy as np

SEED = 20240131

# BMW 320i parameter set used throughout SURVEY.md §8(c)/(d)
VEHICLE = {"length": 4.508, "width": 1.61, "mass": 1093.3, "wb_rear_axle": 1.4227, "a_max": 11.5}

# raw dims / default speeds / buffer factors: reference configurations/simulation/occlusion.yaml:89-114
AGENT_DEFAULTS = {
    "Pedestrian": {"length": 0.3, "width": 0.5, "v": 1.4, "fl": 1.2, "fw": 1.3},
    "Bicycle": {"length": 2.0, "width": 0.9, "v": 5.0, "fl": 1.4, "fw": 2.5},
    "Car": {"length": 4.8, "width": 2.0, "v": 10.0, "fl": 1.2, "fw": 1.3},
    "Truck": {"length": 9.0, "width": 2.5, "v": 10.0, "fl": 1.2, "fw": 1.3},
}

ALL_METRICS = ["hr", "ttc", "be", "ttce", "dce", "wttc", "cp"]
DEFAULT_METRICS = ["hr", "ttc", "ttce", "dce", "wttc", "cp"]  # occlusion.yaml:12-18
DEFAULT_THRESHOLDS = {"harm": 0.1, "risk": 1, "be": None, "cp": None, "ttc": None, "wttc": None,
                      "ttce": None, "dce": None}  # occlusion.yaml:20-28


def _f32(a):
    return np.asarray(a, dtype=np.float64).astype(np.float32).astype(np.float64)


def ego_bundle(n_traj: int, n_states: int, dt: float = 0.1, seed: int = SEED, rng=None) -> np.ndarray:
    """[N, T, 5] (x, y, theta, v, a): constant-acceleration circular arcs from the origin,
    v0 ~ U(0,15), a ~ U(-4,2) (speed clipped at 0), curvature ~ U(-0.1,0.1), heading0 = 0."""
    rng = np.random.default_rng(seed) if rng is None else rng
    v0 = rng.uniform(0.0, 15.0, n_traj)[:, None]
    acc = rng.uniform(-4.0, 2.0, n_traj)[:, None]
    kap = rng.uniform(-0.1, 0.1, n_traj)[:, None]
    kap = np.where(np.abs(kap) < 1e-4, 1e-4, kap)
    t = (np.arange(n_states) * dt)[None, :]
    t_stop = np.where(acc < 0, v0 / np.maximum(-acc, 1e-12), np.inf)
    tc = np.minimum(t, t_stop)
    s = v0 * tc + 0.5 * acc * tc * tc
    v = np.maximum(v0 + acc * tc, 0.0)
    a = np.where(t < t_stop, acc, 0.0) * np.ones_like(t)
    th = kap * s
    x = np.sin(th) / kap
    y = (1.0 - np.cos(th)) / kap
    return _f32(np.stack((x, y, th, v, a), axis=-1))


def agent_table(n_agents: int, n_states: int, dt: float = 0.1, seed: int = SEED + 1, rng=None,
                area=((0.0, 60.0), (-15.0, 15.0)), variance_factor: float = 1.05):
    """List of phantom-agent predictions: 50 % Pedestrian, 25 % Bicycle, 25 % Car, uniform start
    pose, constant velocity, var_k = 0.1 * 1.05^k (reference agent.py:261-280, occlusion.yaml:91)."""
    rng = np.random.default_rng(seed) if rng is None else rng
    kinds = np.array(["Pedestrian", "Pedestrian", "Bicycle", "Car"])
    out = []
    k = np.arange(n_states)
    var = 0.1 * np.power(variance_factor, k)
    for i in range(n_agents):
        kind = str(kinds[i % 4])
        d = AGENT_DEFAULTS[kind]
        x0 = rng.uniform(*area[0])
        y0 = rng.uniform(*area[1])
        yaw = rng.uniform(-np.pi, np.pi)
        yaw = float(_f32(yaw))
        pos = np.stack((x0 + k * dt * d["v"] * np.cos(yaw), y0 + k * dt * d["v"] * np.sin(yaw)), axis=-1)
        out.append({"agent_type": kind, "length": float(_f32(d["length"])), "width": float(_f32(d["width"])),
                    "buf_length": float(_f32(d["length"] * d["fl"])), "buf_width": float(_f32(d["width"] * d["fw"])),
                    "pos": _f32(pos), "yaw": np.full(n_states, yaw), "v": _f32(np.full(n_states, d["v"])),
                    "var": _f32(var)})
    return out


# Every obstacle type of the reference's ObstacleType that the metric core distinguishes (``_lib.KINDS``), with a
# plausible raw length / width / speed and the buffer factors of the nearest kind of AGENT_DEFAULTS.  The car-mass
# kinds keep a buffered area far above the 3.3 m^2 below which -1333.5 + 526.9 size^0.8 is not positive.
VARIED_KINDS = {
    "Pedestrian": AGENT_DEFAULTS["Pedestrian"], "Bicycle": AGENT_DEFAULTS["Bicycle"], "Car": AGENT_DEFAULTS["Car"],
    "Truck": AGENT_DEFAULTS["Truck"],
    "Bus": {"length": 12.0, "width": 2.55, "v": 8.0, "fl": 1.2, "fw": 1.3},
    "Motorcycle": {"length": 2.2, "width": 0.8, "v": 12.0, "fl": 1.4, "fw": 2.5},
    "PriorityVehicle": {"length": 5.2, "width": 2.0, "v": 14.0, "fl": 1.2, "fw": 1.3},
    "ParkedVehicle": {"length": 4.5, "width": 1.8, "v": 0.0, "fl": 1.2, "fw": 1.3},
    "Taxi": {"length": 4.8, "width": 1.9, "v": 9.0, "fl": 1.2, "fw": 1.3},
    "Train": {"length": 30.0, "width": 3.0, "v": 10.0, "fl": 1.2, "fw": 1.3},
    "Unknown": {"length": 1.0, "width": 1.0, "v": 2.0, "fl": 1.2, "fw": 1.3},
}


def varied_agents(n_agents: int, n_states: int, seed: int, *, jitter: bool = False, ragged: bool = True,
                  dt: float = 0.1, area=((-20.0, 50.0), (-25.0, 25.0)), variance_factor: float = 1.05):
    """Case-format predictions that turn, change speed and carry per-axis variances, cycling through every kind of
    VARIED_KINDS.  ``agent_table`` keeps heading, speed and var_x = var_y constant, so a kernel that reads a heading,
    speed or variance from the wrong step or axis agrees with it; these agents tell such mistakes apart.

    * kinematic (default): heading yaw0 + w t with w ~ U(-0.6, 0.6) rad/s, speed max(v0 + a t, 0) with
      a ~ U(-3, 2) (ParkedVehicle: 0), positions integrated from both; every third agent starts within 0.15 rad of
      +-pi and turns outwards, so its heading leaves [-pi, pi].
    * ``jitter``: heading, speed and variances drawn independently per step, positions a random walk -- any index
      offset then gives a large error, not a second-order one.
    * per state var_x, var_y = 0.1 * 1.05^k * U(0.3, 3) each, both zero on about 10 % of the states, carried as a
      diagonal ``cov`` [T_a, 2, 2] (``var`` is var_x).
    * ``ragged``: every fifth agent has 1, 2, 8, 9 or n_states + 20 (at most 128) states instead of n_states.
    All values are float32-representable."""
    rng = np.random.default_rng(seed)
    kinds = list(VARIED_KINDS)
    out = []
    for i in range(n_agents):
        kind = kinds[i % len(kinds)]
        d = VARIED_KINDS[kind]
        n = n_states
        if ragged and i % 5 == 4:
            n = [1, 2, 8, 9, min(n_states + 20, 128)][(i // 5) % 5]
        t = np.arange(n) * dt
        x0, y0 = rng.uniform(*area[0]), rng.uniform(*area[1])
        if i % 3 == 0:
            sgn = rng.choice((-1.0, 1.0))
            yaw0, w = sgn * (np.pi - rng.uniform(0.0, 0.15)), sgn * rng.uniform(0.2, 0.6)
        else:
            yaw0, w = rng.uniform(-np.pi, np.pi), rng.uniform(-0.6, 0.6)
        if jitter:
            yaw = yaw0 + rng.uniform(-1.5, 1.5, n)
            v = rng.uniform(0.0, 1.5 * d["v"] + 0.5, n) * (d["v"] > 0)
            x = x0 + np.cumsum(rng.normal(0.0, 0.4, n))
            y = y0 + np.cumsum(rng.normal(0.0, 0.4, n))
        else:
            yaw = yaw0 + w * t
            v = np.maximum(d["v"] + rng.uniform(-3.0, 2.0) * t, 0.0) * (d["v"] > 0)   # a parked vehicle stays
            x = x0 + np.concatenate(([0.0], np.cumsum(v[:-1] * np.cos(yaw[:-1]) * dt)))
            y = y0 + np.concatenate(([0.0], np.cumsum(v[:-1] * np.sin(yaw[:-1]) * dt)))
        base = 0.1 * np.power(variance_factor, np.arange(n))
        vx, vy = _f32(base * rng.uniform(0.3, 3.0, n)), _f32(base * rng.uniform(0.3, 3.0, n))
        zero = rng.random(n) < 0.1
        vx[zero] = vy[zero] = 0.0
        cov = np.zeros((n, 2, 2))
        cov[:, 0, 0], cov[:, 1, 1] = vx, vy
        out.append({"agent_type": kind, "length": float(_f32(d["length"])), "width": float(_f32(d["width"])),
                    "buf_length": float(_f32(d["length"] * d["fl"])), "buf_width": float(_f32(d["width"] * d["fw"])),
                    "pos": _f32(np.stack((x, y), -1)), "yaw": _f32(yaw), "v": _f32(v), "var": vx, "cov": cov})
    return out


def rotate_bundle(ego: np.ndarray, seed: int) -> np.ndarray:
    """``ego`` [N, T, 5] with every trajectory turned about the origin by its own heading ~ U(-pi, pi): the arcs of
    ``ego_bundle`` all start along +x, so their collision-probability boxes mostly travel along x; turned, both axes
    of an agent's covariance matter."""
    ego = np.asarray(ego, dtype=np.float64)
    h = np.random.default_rng(seed).uniform(-np.pi, np.pi, len(ego))[:, None]
    c, s = np.cos(h), np.sin(h)
    out = ego.copy()
    out[..., 0] = c * ego[..., 0] - s * ego[..., 1]
    out[..., 1] = s * ego[..., 0] + c * ego[..., 1]
    out[..., 2] = ego[..., 2] + h
    return _f32(out)


def make_case(n_traj: int, n_agents: int, n_states: int, dt: float = 0.1, seed: int = SEED,
              activated_metrics=None, thresholds=None, agent_states: int | None = None):
    """A complete *case* (see ``oracle/ref_runner.py`` for the format)."""
    rng = np.random.default_rng(seed)
    ego = ego_bundle(n_traj, n_states, dt, rng=rng)
    agents = agent_table(n_agents, agent_states or n_states, dt, rng=rng)
    return {"dt": dt, "vehicle": {k: float(_f32(v)) for k, v in VEHICLE.items()}, "ego": ego, "agents": agents,
            "activated_metrics": list(ALL_METRICS if activated_metrics is None else activated_metrics),
            "thresholds": dict(DEFAULT_THRESHOLDS if thresholds is None else thresholds)}


def make_varied_case(n_traj: int, n_agents: int, n_states: int, dt: float = 0.1, seed: int = SEED,
                     activated_metrics=None, thresholds=None, *, jitter: bool = False, **agent_kw):
    """``make_case`` with its trajectories turned by ``rotate_bundle`` and ``varied_agents`` for its agents."""
    case = make_case(n_traj, 0, n_states, dt, seed, activated_metrics, thresholds)
    case["ego"] = rotate_bundle(case["ego"], seed)
    case["agents"] = varied_agents(n_agents, n_states, seed, jitter=jitter, dt=dt, **agent_kw)
    return case


# named BASELINE.json configurations -----------------------------------------------------------
C_LAT = {"name": "C-lat", "n_traj": 1000, "n_agents": 32, "n_states": 31}
C_SWEEP = {"name": "C-sweep", "n_traj": 1_000_000, "n_agents": 256, "n_states": 51}
C_VIS = {"name": "C-vis", "n_rays": 4096, "n_obstacles": 512, "n_frames": 10_000}


def obstacle_frames(n_frames: int, n_obstacles: int, seed: int = SEED + 2, half_extent: float = 50.0,
                    length: float = 4.8, width: float = 2.0):
    """C-vis input: per frame ``n_obstacles`` rectangles (cx, cy, yaw, half_len, half_wid) uniform in
    the 100 m x 100 m square around the ego at the origin -> float32 [F, O, 5]."""
    rng = np.random.default_rng(seed)
    rect = np.empty((n_frames, n_obstacles, 5), dtype=np.float32)
    rect[..., 0] = rng.uniform(-half_extent, half_extent, (n_frames, n_obstacles))
    rect[..., 1] = rng.uniform(-half_extent, half_extent, (n_frames, n_obstacles))
    rect[..., 2] = rng.uniform(-np.pi, np.pi, (n_frames, n_obstacles))
    rect[..., 3] = 0.5 * length
    rect[..., 4] = 0.5 * width
    return rect
