"""Oracle B: vectorised float64 numpy restatement of the dense metric core (TEST INFRASTRUCTURE).

Restates, for a whole trajectory bundle at once, what the reference computes one trajectory at a
time in ``Metric.evaluate_metrics`` (``frenetix_occlusion/metrics/metric.py:35-100``).  Every
function cites the reference lines it follows.  It is cross-checked against oracle A (the
reference's own modules run verbatim over shims, ``oracle/ref_runner.py``) through the committed
fixtures in ``tests/golden`` -- masks/indices exactly, floats to 1e-12.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may import this.
"""
from __future__ import annotations

import json
import os

import numpy as np
from scipy.special import ndtr

from .geometry import obb_distance, obb_intersects

# harm coefficients actually read on this path (reference frenetix_occlusion/config/harm_params.json,
# keys log_reg.reduced_sym_angle_areas, log_reg.ignore_angle, pedestrian; SURVEY.md §8a M7)
HARM_COEFFS = {
    "reduced_sym": {"const": -4.457, "speed": 0.177, "side": 0.244, "rear": -0.431},
    "ignore_angle": {"const": -4.591, "speed": 0.185},
    "pedestrian": {"const": 3.164, "speed": 0.288},
}

# obstacle_protection, harm_model.py:15-32 (keyed by ObstacleType string value)
PROTECTED = {"car": True, "truck": True, "bus": True, "bicycle": False, "pedestrian": False,
             "priorityvehicle": True, "parkedvehicle": True, "train": True, "motorcycle": False,
             "taxi": True, "unknown": False}


def obstacle_mass(agent_type: str, size: float) -> float:
    """harm_model.py:158-190 (``size`` = buffered length*width, harm_model.py:73)."""
    t = agent_type.lower()
    if t in ("car", "priorityvehicle", "parkedvehicle", "taxi"):
        return -1333.5 + 526.9 * np.power(size, 0.8)
    return {"truck": 25000.0, "bus": 13000.0, "bicycle": 90.0, "pedestrian": 75.0, "train": 118800.0,
            "motorcycle": 250.0}.get(t, 0.0)


def check_required_metrics(metric_names):
    """metric.py:125-147 -- dependency ordering (returns a new list)."""
    m = list(metric_names)
    if "wttc" in m:
        if "ttc" in m:
            m.remove("ttc")
        m.insert(0, "ttc")
    if "ttc" in m or "ttce" in m or "be" in m:
        if "dce" in m:
            m.remove("dce")
        m.insert(0, "dce")
    if "hr" in m:
        if "cp" in m:
            m.remove("cp")
        m.insert(0, "cp")
    known = {"dce", "cp", "ttc", "ttce", "wttc", "be", "hr"}
    return [x for x in m if x in known]


# --------------------------------------------------------------------------------------------
def _stack_agents(case):
    """``var`` [A, Tm, 2] holds (sigma_x^2, sigma_y^2) of every state: the diagonal of the agent's ``cov``
    (``cov_list``, [T_a, 2, 2]) when it has one, else its scalar ``var`` on both axes."""
    ags = case["agents"]
    A = len(ags)
    Ta = np.array([len(np.asarray(a["yaw"])) for a in ags], dtype=np.int64)
    Tm = int(Ta.max()) if A else 0
    pos = np.zeros((A, Tm, 2))
    yaw = np.zeros((A, Tm))
    vel = np.zeros((A, Tm))
    var = np.full((A, Tm, 2), 0.1)
    for k, a in enumerate(ags):
        pos[k, :Ta[k]] = np.asarray(a["pos"], dtype=np.float64).reshape(-1, 2)
        yaw[k, :Ta[k]] = a["yaw"]
        vel[k, :Ta[k]] = a["v"]
        if "cov" in a:
            c = np.asarray(a["cov"], dtype=np.float64)
            var[k, :Ta[k]] = np.stack((c[:, 0, 0], c[:, 1, 1]), -1)
        else:
            var[k, :Ta[k]] = np.asarray(a["var"], dtype=np.float64)[:, None]
    return A, Ta, Tm, pos, yaw, vel, var


def collision_probability(case):
    """CP per step, [N, A, T-1].  collision_probability.py:14-126 (see SURVEY.md appendix A):
    ego state i pairs with agent position i-1, agent yaw i, covariance i-1; 5 m strict gate on the
    min distance of the three obstacle points to the raw ego point; three axis-aligned ego boxes.
    sigma_x, sigma_y = sqrt(cov[i-1][0][0]), sqrt(cov[i-1][1][1]) (mvnun with a diagonal covariance factorises
    per axis); a correlated ``cov`` is ``tests/corr_oracle.py``'s case and raises here."""
    for k, a in enumerate(case["agents"]):
        if "cov" in a and np.any(np.asarray(a["cov"])[:, [0, 1], [1, 0]] != 0):
            raise ValueError(f"agent {k}: correlated covariance (not a diagonal one)")
    ego = np.asarray(case["ego"], dtype=np.float64)
    N, T, _ = ego.shape
    A, Ta, Tm, pos, yaw, vel, var = _stack_agents(case)
    L, W = case["vehicle"]["length"], case["vehicle"]["width"]
    cp = np.zeros((N, A, max(T - 1, 0)))
    inside = np.zeros((N, A, max(T - 1, 0)), dtype=bool)
    gate_margin = np.full((N, A, max(T - 1, 0)), np.inf)   # |min distance - 5.0| (tie diagnostics)
    for a in range(A):
        nmax = min(T, Ta[a])          # i < len(mean_list)
        if nmax < 2:
            continue
        i = np.arange(1, nmax)
        lb = case["agents"][a]["buf_length"]
        p = pos[a, i - 1]                                             # :52  mean_list[:min_len-1]
        h = np.stack((np.cos(yaw[a, i]), np.sin(yaw[a, i])), -1) * lb / 2   # :51  yaw_list[1:min_len]
        mus = np.stack((p, p + h, p - h), 0)                          # [3, n, 2]
        e = ego[:, i, 0:2]                                            # [N, n, 2] raw rear-axle point
        d = np.sqrt(((mus[None] - e[:, None]) ** 2).sum(-1))         # [N, 3, n]
        gate = d.min(1) > 5.0                                         # :65-67 strict
        v = var[a, i - 1].copy()                                      # [n, 2]
        v[(v == 0.0).all(-1)] = 0.1                                   # :85-87 (an all-zero matrix)
        sig = np.sqrt(v)
        th = ego[:, i, 2]
        off = np.stack((np.cos(th), np.sin(th)), -1) * (L / 3.0)      # r_x*(2/3)*a_x, :160-162
        cen = np.stack((e, e + off, e - off), 1)                      # [N, 3, n, 2]
        half = np.array([L / 6.0, W / 2.0])                           # :35
        lo = cen - half
        hi = cen + half
        # [N, mu(3), box(3), n, 2]
        zhi = (hi[:, None] - mus[None, :, None]) / sig[None, None, None]
        zlo = (lo[:, None] - mus[None, :, None]) / sig[None, None, None]
        pr = ndtr(zhi) - ndtr(zlo)
        prob = (pr[..., 0] * pr[..., 1]).sum((1, 2)) / 3.0            # :115-122
        cp[:, a, i - 1] = np.where(gate, 0.0, prob)
        inside[:, a, i - 1] = ~gate
        gate_margin[:, a, i - 1] = np.abs(d.min(1) - 5.0)
    return cp, inside, gate_margin


def dce_metric(case):
    """DCE per pair.  dce.py:52-99 + convert_dynamic_obstacle.py:17-86: ego rectangle centred at the
    axle-shifted point, agent rectangle = *unbuffered* agent.shape, same-step pairing over
    i in [0, min(T_e, T_a)), distances rounded to 3 decimals, strict-min + first index.
    Also returns the unrounded per-step distances [N, A, T] (nan where the agent has no state)."""
    ego = np.asarray(case["ego"], dtype=np.float64)
    N, T, _ = ego.shape
    A, Ta, Tm, pos, yaw, vel, var = _stack_agents(case)
    vp = case["vehicle"]
    cx = ego[..., 0] + vp["wb_rear_axle"] * np.cos(ego[..., 2])      # :73
    cy = ego[..., 1] + vp["wb_rear_axle"] * np.sin(ego[..., 2])
    dist = np.full((N, A, T), np.nan)
    for a in range(A):
        n = min(T, Ta[a])
        ag = case["agents"][a]
        dist[:, a, :n] = obb_distance(cx[:, :n], cy[:, :n], ego[:, :n, 2], vp["length"] / 2, vp["width"] / 2,
                                      pos[a, :n, 0][None], pos[a, :n, 1][None], yaw[a, :n][None],
                                      ag["length"] / 2, ag["width"] / 2)
    r = np.round(dist, 3)                                            # :79
    rr = np.where(np.isnan(r), np.inf, r)
    dce = rr.min(-1)
    time_dce = np.where(np.isinf(dce), 0, rr.argmin(-1))             # first minimum; (inf, 0) if T_a == 0
    return dce, time_dce.astype(np.int64), dist


def harm_model(case):
    """Harm per step, ego and obstacle, [N, A, T-1] (nan beyond P_a = min(T_e-1, T_a)).
    harm_model.py:35-107, logistic_regression.py:11-75.  Impact angles are NOT wrapped."""
    ego = np.asarray(case["ego"], dtype=np.float64)
    N, T, _ = ego.shape
    A, Ta, Tm, pos, yaw, vel, var = _stack_agents(case)
    m_e = case["vehicle"]["mass"]
    eh = np.full((N, A, max(T - 1, 0)), np.nan)
    oh = np.full((N, A, max(T - 1, 0)), np.nan)
    ang_margin = np.full((N, A, max(T - 1, 0)), np.inf)
    C = HARM_COEFFS
    t_a = 45 / 180 * np.pi
    t_b = 3 * t_a

    def lr4s(v, ang):
        c = np.where((-t_a < ang) & (ang < t_a), 0.0,
                     np.where(((t_a <= ang) & (ang < t_b)) | ((-t_a >= ang) & (ang > -t_b)),
                              C["reduced_sym"]["side"], C["reduced_sym"]["rear"]))
        return 1.0 / (1.0 + np.exp(-C["reduced_sym"]["const"] - C["reduced_sym"]["speed"] * v - c))

    for a in range(A):
        ag = case["agents"][a]
        P = min(T - 1, Ta[a])                                         # :67
        if P == 0:
            continue
        t = np.arange(P)
        typ = ag["agent_type"].lower()
        m_o = obstacle_mass(typ, ag["buf_length"] * ag["buf_width"])  # :73,78
        th, x, y, v = ego[:, t, 2], ego[:, t, 0], ego[:, t, 1], ego[:, t, 3]
        pdof = yaw[a, t][None] - th + np.pi                           # :81
        rel = np.arctan2(pos[a, t, 1][None] - y, pos[a, t, 0][None] - x)  # :82-83
        ang_e = rel - th                                              # :86
        ang_o = np.pi + rel - yaw[a, t][None]                         # :88
        dv = np.sqrt(v ** 2 + vel[a, t][None] ** 2 + 2 * v * vel[a, t][None] * np.cos(pdof))  # :91-95
        dv_e = m_o / (m_e + m_o) * dv                                 # :96
        dv_o = m_e / (m_e + m_o) * dv                                 # :97
        prot = PROTECTED.get(typ)
        if prot is True:                                              # harm_model.py:125-131
            eh[:, a, :P] = lr4s(dv_e, ang_e)
            oh[:, a, :P] = lr4s(dv_o, ang_o)
            mg = np.inf
            for b in (-t_b, -t_a, t_a, t_b):
                mg = np.minimum(mg, np.minimum(np.abs(ang_e - b), np.abs(ang_o - b)))
            ang_margin[:, a, :P] = mg
        elif prot is False:                                           # :133-146
            eh[:, a, :P] = 1.0 / (1.0 + np.exp(-C["ignore_angle"]["const"] - C["ignore_angle"]["speed"] * dv_e))
            oh[:, a, :P] = 1.0 / (1.0 + np.exp(C["pedestrian"]["const"] - C["pedestrian"]["speed"] * dv_o))
        else:
            eh[:, a, :P] = 1.0
            oh[:, a, :P] = 1.0
    return eh, oh, ang_margin


def _np_interp_ref(xq, xp, fp):
    """``scipy.interpolate.interp1d(xp, fp, kind='linear')`` for 1-D float64 delegates to
    ``numpy.interp`` (scipy ``_call_linear_np``) after a bounds check that raises ValueError."""
    if np.any(xq < xp[0]) or np.any(xq > xp[-1]):
        raise ValueError("interp1d bounds")
    return np.interp(xq, xp, fp)


def brake_evaluation(case, ttc):
    """BE per pair.  be.py:31-193.  Returns (required_constant_deceleration [N,A], btn [N,A],
    error [N] -- True where the reference raises ValueError from interp1d)."""
    ego = np.asarray(case["ego"], dtype=np.float64)
    N, T, _ = ego.shape
    A, Ta, Tm, pos, yaw, vel, var = _stack_agents(case)
    vp = case["vehicle"]
    dt = case["dt"]
    rcd = np.zeros((N, A))
    err = np.zeros(N, dtype=bool)
    pairs = np.argwhere(np.isfinite(ttc) & (ttc > 0))               # :49-50
    for n in np.unique(pairs[:, 0]) if len(pairs) else []:
        x, y, th, v, acc = (ego[n, :, k] for k in range(5))
        dist = np.insert(np.cumsum(np.sqrt(np.diff(x) ** 2 + np.diff(y) ** 2)), 0, 0)   # :99
        time = np.arange(T - 1) * dt                                   # :102
        for a in pairs[pairs[:, 0] == n][:, 1]:
            ag = case["agents"][a]
            lo = np.round(abs(min(min(acc), 0)), 2)                    # :68
            hi = 5
            cur = None
            nn = min(T, Ta[a])
            try:
                for _ in range(10):                                    # :69
                    cur = (lo + hi) / 2
                    v_new = np.insert(np.maximum(v[1] - cur * time, 0), 0, v[0:1])      # :109
                    dist_new = np.insert(np.cumsum(v_new * dt), 0, 0)[:-1]              # :113
                    xn = _np_interp_ref(dist_new, dist, x)                               # :116-124
                    yn = _np_interp_ref(dist_new, dist, y)
                    tn = _np_interp_ref(dist_new, dist, th)
                    cxn = xn + vp["wb_rear_axle"] * np.cos(tn)
                    cyn = yn + vp["wb_rear_axle"] * np.sin(tn)
                    hit = obb_intersects(cxn[:nn], cyn[:nn], tn[:nn], vp["length"] / 2, vp["width"] / 2,
                                         pos[a, :nn, 0], pos[a, :nn, 1], yaw[a, :nn],
                                         ag["length"] / 2, ag["width"] / 2)
                    if nn > 0 and not hit.any():                       # :74-75 ("0 in collisions")
                        hi = cur
                    else:
                        lo = cur
                    if hi - lo < 0.1:                                  # :79
                        break
                rcd[n, a] = cur
            except ValueError:
                err[n] = True
    btn = rcd / vp["a_max"]                                           # :56
    return rcd, btn, err


def evaluate_bundle(case, want_detail: bool = True):
    """Everything ``Metric.evaluate_metrics`` yields, for all N trajectories at once.

    Returns a dict of arrays; keys are only present for metrics that ran (after
    ``check_required_metrics``).  ``valid`` restates the threshold logic of metric.py:50-98,
    ``be_error`` marks trajectories on which the reference raises."""
    order = check_required_metrics(case["activated_metrics"])
    thr = case["thresholds"]
    ego = np.asarray(case["ego"], dtype=np.float64)
    N, T, _ = ego.shape
    A = len(case["agents"])
    out = {"order": order, "N": N, "A": A, "T": T}
    valid = np.ones(N, dtype=bool)
    if A == 0 or not order:                                          # metric.py:44-45
        out["valid"] = valid
        out["be_error"] = np.zeros(N, dtype=bool)
        return out
    Ta = np.array([len(np.asarray(a["yaw"])) for a in case["agents"]])
    if "cp" in order:
        cp, inside, gate_margin = collision_probability(case)
        out["cp"] = cp
        if want_detail:
            out["gate_margin"] = gate_margin
        out["gate_fraction"] = float(inside.mean()) if inside.size else 0.0
    if "dce" in order:
        dce, tdce, dist = dce_metric(case)
        out["dce"], out["time_dce"] = dce, tdce
        if want_detail:
            out["dist"] = dist
    if "ttc" in order:
        if "dce" not in out:
            raise ValueError("DCE is not available in results, but is needed to evaluate TTC metric!")
        out["ttc"] = np.where(np.isclose(out["dce"], 0.0), np.round(out["time_dce"] * case["dt"], 3), np.inf)  # ttc.py:40-46
    if "ttce" in order:
        out["ttce"] = np.round(out["time_dce"] * case["dt"], 3)       # ttce.py:39
    if "wttc" in order:
        out["wttc"] = out["ttc"].min(1)                               # wttc.py:32-42
    if "hr" in order:
        cp = out["cp"]
        eh, oh, ang_margin = harm_model(case)
        P = np.minimum(T - 1, Ta)
        has = P > 0                                                   # harm_model.py:68-70 (skipped pairs)
        er = eh * cp                                                  # hr.py:78-79 (nan beyond P)
        orr = oh * cp
        pair = {}
        with np.errstate(invalid="ignore"), __import__("warnings").catch_warnings():
            __import__("warnings").simplefilter("ignore")
            pair["max_ego_risk"] = np.nanmax(np.where(has[None, :, None], er, 0.0), -1)
            pair["max_obst_risk"] = np.nanmax(np.where(has[None, :, None], orr, 0.0), -1)
            pair["max_obst_risk_index"] = np.argmax(np.where(np.isnan(orr), -np.inf, orr), -1)
            pair["max_ego_harm"] = np.nanmax(np.where(has[None, :, None], eh, 0.0), -1)
            pair["max_obst_harm"] = np.nanmax(np.where(has[None, :, None], oh, 0.0), -1)
        mcp = cp.max(-1)                                              # hr.py:81 np.max over the full cp vector
        amax = cp.argmax(-1)
        # hr.py:82 obst_harm_traj[key][argmax(cp)]; cp is zero for i >= T_a so argmax < P whenever max > 0.01
        ohc = np.take_along_axis(np.nan_to_num(oh, nan=0.0), amax[..., None], -1)[..., 0]
        pair["max_obst_harm_with_cp"] = np.where(mcp > 0.01, ohc, 0.0)
        pair["max_collision_probability"] = mcp
        for k in pair:
            pair[k] = np.where(has[None, :], pair[k], 0)
        out["hr_pair"] = pair
        out["hr_has"] = has
        if want_detail:
            out["ego_harm"], out["obst_harm"] = eh, oh
            out["ego_risk"], out["obst_risk"] = er, orr
            out["angle_margin"] = ang_margin
        for k_all, k_pair in (("max_ego_risk_all", "max_ego_risk"), ("max_obst_risk_all", "max_obst_risk"),
                              ("max_ego_harm_all", "max_ego_harm"), ("max_obst_harm_all", "max_obst_harm"),
                              ("max_collision_probability_all", "max_collision_probability"),
                              ("max_obst_harm_with_cp_all", "max_obst_harm_with_cp")):
            out[k_all] = np.maximum(pair[k_pair].max(1), 0.0)        # hr.py:69-74 init 0
    be_err = np.zeros(N, dtype=bool)
    if "be" in order:
        if "ttc" not in out:
            raise KeyError("ttc")                                    # be.py:39
        rcd, btn, be_err = brake_evaluation(case, out["ttc"])
        out["be_rcd"], out["be_btn"] = rcd, btn
    out["be_error"] = be_err
    # ---- thresholds, metric.py:50-98 (strict comparisons, None disables) -----------------------
    if "be" in order and thr.get("be") is not None:
        valid &= ~(out["be_btn"] > thr["be"]).any(1)
    if "hr" in order and thr.get("harm") is not None:
        valid &= ~(out["max_obst_harm_with_cp_all"] > thr["harm"])
    if "hr" in order and thr.get("risk") is not None:
        valid &= ~(out["max_obst_risk_all"] > thr["risk"])
    if "hr" in order and thr.get("cp") is not None:
        valid &= ~(out["max_collision_probability_all"] > thr["cp"])
    if "ttc" in order and thr.get("ttc") is not None:
        valid &= ~(out["ttc"].min(1) < thr["ttc"])
    if "dce" in order and thr.get("dce") is not None:
        valid &= ~(out["dce"] < thr["dce"]).any(1)
    out["valid"] = valid
    return out


def to_reference_dict(out, n, case):
    """Re-assemble trajectory ``n``'s results in the reference's nested-dict shape (SURVEY.md §8b),
    keyed by the prediction ids oracle A uses (``int(str(10000+k)+'0')``)."""
    pids = [int(str(10000 + k) + "0") for k in range(out["A"])]
    T = out["T"]
    Ta = [len(np.asarray(a["yaw"])) for a in case["agents"]]
    res = {}
    for name in out["order"]:
        if name == "cp":
            res["cp"] = {p: out["cp"][n, k] for k, p in enumerate(pids)}
        elif name == "dce":
            res["dce"] = {p: {"dce": out["dce"][n, k], "time_dce": int(out["time_dce"][n, k])} for k, p in enumerate(pids)}
        elif name == "ttc":
            res["ttc"] = {p: out["ttc"][n, k] for k, p in enumerate(pids)}
        elif name == "ttce":
            res["ttce"] = {p: out["ttce"][n, k] for k, p in enumerate(pids)}
        elif name == "wttc":
            res["wttc"] = out["wttc"][n]
        elif name == "be":
            res["be"] = {p: {"required_constant_deceleration": out["be_rcd"][n, k],
                             "break_threat_number": out["be_btn"][n, k]} for k, p in enumerate(pids)}
        elif name == "hr":
            hr = {}
            for k, p in enumerate(pids):
                if not out["hr_has"][k]:
                    continue
                P = min(T - 1, Ta[k])
                hr[p] = {"max_ego_risk": out["hr_pair"]["max_ego_risk"][n, k],
                         "max_obst_risk": out["hr_pair"]["max_obst_risk"][n, k],
                         "max_obst_harm_with_cp": out["hr_pair"]["max_obst_harm_with_cp"][n, k],
                         "max_obst_risk_index": int(out["hr_pair"]["max_obst_risk_index"][n, k]),
                         "max_ego_harm": out["hr_pair"]["max_ego_harm"][n, k],
                         "max_obst_harm": out["hr_pair"]["max_obst_harm"][n, k],
                         "ego_risk_traj": out["ego_risk"][n, k, :P], "obst_risk_traj": out["obst_risk"][n, k, :P],
                         "ego_harm_traj": out["ego_harm"][n, k, :P], "obst_harm_traj": out["obst_harm"][n, k, :P],
                         "collision_probability": out["cp"][n, k],
                         "max_collision_probability": out["hr_pair"]["max_collision_probability"][n, k]}
            for k_all in ("max_ego_risk_all", "max_obst_risk_all", "max_ego_harm_all", "max_obst_harm_all",
                          "max_collision_probability_all", "max_obst_harm_with_cp_all"):
                hr[k_all] = out[k_all][n]
            res["hr"] = hr
    return res


def load_case_json(path):
    with open(path) as f:
        d = json.load(f)
    case = d["case"]
    case["ego"] = np.asarray(case["ego"], dtype=np.float64)
    for a in case["agents"]:
        for k in ("pos", "yaw", "v", "var"):
            a[k] = np.asarray(a[k], dtype=np.float64)
    return case, d.get("reference"), d.get("order")


def case_to_json(case):
    c = dict(case)
    c["ego"] = np.asarray(case["ego"]).tolist()
    c["agents"] = [{k: (np.asarray(v).tolist() if k in ("pos", "yaw", "v", "var") else v) for k, v in a.items()}
                   for a in case["agents"]]
    return c
