"""CUDA-vs-oracle comparison for the dense metric core (used by the -m gpu tests and the report
script).  Tolerances follow BASELINE.json's north_star: floating-point metrics within 1e-4
relative (fp32 kernel vs float64 oracle) with a small absolute floor; validity masks and discrete
indices bit-exact except *documented exact-threshold ties*, which are recognised from the float64
oracle's own margins and counted:

* DCE rounding tie: ``np.round(d, 3)`` of a step whose unrounded distance lies within TIE_DIST of a
  rounding boundary (x.xxx5) and which competes for the minimum -> dce may move by 0.001 and
  time_dce may move to another step.
* LR4S class tie: an (un-wrapped) impact angle within TIE_ANG of +-pi/4 / +-3pi/4.
* CP gate tie: min obstacle-point distance within TIE_GATE of the 5.0 m gate.
* BE bisection tie: the float32 intersection test flips at one bisection probe -> the returned
  midpoint moves by one bisection level; also the interp1d range check (FO_F_BE_RANGE).
"""
import numpy as np

RTOL = 1e-4
ATOL_CP = 2e-7       # cp / risk absolute floor (reference emits exact 0.0 next to 1e-12-scale values)
ATOL_HARM = 1e-6
TIE_DIST = 5e-5      # metres from a rounding boundary
TIE_ANG = 2e-5       # radians from an LR4S class boundary
TIE_GATE = 2e-5      # metres from the 5 m gate


def _close(g, r, rtol, atol):
    return np.isclose(g, r, rtol=rtol, atol=atol, equal_nan=True)


def compare_bundle(out, res, case):
    """``out``: oracle.metric_oracle.evaluate_bundle(case); ``res``: dict of numpy arrays from the GPU
    (valid, summary, flags, pair, step).  Returns a report dict with hard failures and tie counts."""
    rep = {"fail": [], "ties": {}, "n_pairs": out["N"] * out["A"]}
    order = out["order"]
    N, A, T = out["N"], out["A"], out["T"]
    pair, step, summ = res.get("pair"), res.get("step"), res["summary"]
    ok_traj = ~out["be_error"]
    gpu_err = (res["flags"] & 1).astype(bool)
    bad_flag = gpu_err != out["be_error"]
    rep["ties"]["be_range_flag"] = int(bad_flag.sum())
    ok_traj &= ~gpu_err
    tie_traj = bad_flag.copy()          # trajectories whose mask may legitimately differ

    if A == 0 or not order:
        if not res["valid"].all():
            rep["fail"].append("valid must be all-true without agents/metrics")
        return rep

    # ---------------------------------------------------------------- DCE / TTC
    dce_tie_pair = np.zeros((N, A), dtype=bool)
    if "dce" in order:
        dist = out["dist"]
        frac = np.abs(dist * 1000.0 - np.floor(dist * 1000.0) - 0.5) / 1000.0
        near = (frac < TIE_DIST) & (np.round(dist, 3) <= out["dce"][..., None] + 0.0011)
        dce_tie_pair = np.nan_to_num(near, nan=0).astype(bool).any(-1)
        if pair is not None:
            g_dce = np.round(pair[..., 0].astype(np.float64), 3)
            g_t = pair[..., 1].astype(np.int64)
            bad = ~((g_dce == out["dce"]) & (g_t == out["time_dce"]))
            hard = bad & ~dce_tie_pair
            hard &= ok_traj[:, None]
            rep["ties"]["dce_round"] = int((bad & dce_tie_pair).sum())
            if hard.any():
                i = np.argwhere(hard)[0]
                rep["fail"].append(f"dce/time_dce mismatch at {tuple(i)}: gpu ({g_dce[tuple(i)]}, {g_t[tuple(i)]}) "
                                   f"oracle ({out['dce'][tuple(i)]}, {out['time_dce'][tuple(i)]}); {int(hard.sum())} pairs")
            if (np.abs(g_dce - out["dce"])[bad & dce_tie_pair] > 0.0011).any():
                rep["fail"].append("dce tie moved by more than one rounding step")
        g_min = np.round(summ[:, 6].astype(np.float64), 3)
        o_min = out["dce"].min(1)
        bad = (g_min != o_min) & ~dce_tie_pair.any(1)
        if bad.any():
            rep["fail"].append(f"summary min_dce mismatch on {int(bad.sum())} trajectories")
        tie_traj |= dce_tie_pair.any(1) & (("dce" in order and case["thresholds"].get("dce") is not None)
                                           or (np.abs(out["dist"]) < 0.001).any((1, 2)))
    if "wttc" in order or "ttc" in order:
        o_w = out["ttc"].min(1)
        g_w = np.round(summ[:, 7].astype(np.float64), 3)
        bad = (g_w != o_w) & ok_traj & ~dce_tie_pair.any(1)
        if bad.any():
            i = int(np.argmax(bad))
            rep["fail"].append(f"wttc mismatch at traj {i}: gpu {g_w[i]} oracle {o_w[i]} ({int(bad.sum())})")

    # ---------------------------------------------------------------- CP
    cp_tie_pair = np.zeros((N, A), dtype=bool)
    if "cp" in order:
        gate_tie = out["gate_margin"] < TIE_GATE
        cp_tie_pair = gate_tie.any(-1)
        if step is not None:
            bad = ~_close(step[..., 0], out["cp"], RTOL, ATOL_CP)
            rep["ties"]["cp_gate"] = int((bad & gate_tie).sum())
            hard = bad & ~gate_tie
            if hard.any():
                i = tuple(np.argwhere(hard)[0])
                rep["fail"].append(f"cp mismatch at {i}: gpu {step[..., 0][i]!r} oracle {out['cp'][i]!r} "
                                   f"({int(hard.sum())} of {hard.size})")
            rep["cp_max_rel"] = float(np.max(np.abs(step[..., 0] - out["cp"]) / np.maximum(out["cp"], 1e-3)))

    # ---------------------------------------------------------------- HR
    if "hr" in order:
        ang_tie = out["angle_margin"] < TIE_ANG
        hr_tie_pair = ang_tie.any(-1) | cp_tie_pair
        if step is not None:
            for col, name in ((1, "ego_harm"), (2, "obst_harm")):
                bad = ~_close(step[..., col], out[name], RTOL, ATOL_HARM)
                rep["ties"]["lr4s_" + name] = int((bad & ang_tie).sum())
                hard = bad & ~ang_tie
                if hard.any():
                    i = tuple(np.argwhere(hard)[0])
                    rep["fail"].append(f"{name} mismatch at {i}: gpu {step[..., col][i]!r} oracle {out[name][i]!r} "
                                       f"({int(hard.sum())})")
        if pair is not None:
            cols = {"max_ego_risk": (2, ATOL_CP), "max_obst_risk": (3, ATOL_CP), "max_obst_harm_with_cp": (5, ATOL_HARM),
                    "max_ego_harm": (6, ATOL_HARM), "max_obst_harm": (7, ATOL_HARM),
                    "max_collision_probability": (8, ATOL_CP)}
            for name, (col, atol) in cols.items():
                bad = ~_close(pair[..., col], out["hr_pair"][name], RTOL, atol) & ~hr_tie_pair
                if name == "max_obst_harm_with_cp":   # 0.01 floor / argmax ties between near-equal cp values
                    mcp = out["hr_pair"]["max_collision_probability"]
                    floor_tie = np.abs(mcp - 0.01) < 1e-5
                    srt = np.sort(out["cp"], -1)
                    arg_tie = (srt[..., -1] - srt[..., -2]) < 1e-4 * np.maximum(srt[..., -1], 1e-30) if out["cp"].shape[-1] > 1 \
                        else np.zeros_like(floor_tie)
                    rep["ties"]["harm_with_cp"] = int((bad & (floor_tie | arg_tie)).sum())
                    bad &= ~(floor_tie | arg_tie)
                if bad.any():
                    i = tuple(np.argwhere(bad)[0])
                    rep["fail"].append(f"pair {name} mismatch at {i}: gpu {pair[..., col][i]!r} "
                                       f"oracle {out['hr_pair'][name][i]!r} ({int(bad.sum())})")
            idx_bad = (pair[..., 4].astype(np.int64) != out["hr_pair"]["max_obst_risk_index"]) & ~hr_tie_pair
            if idx_bad.any():
                real = idx_bad & ~risk_index_tie(out, pair[..., 4].astype(np.int64))
                rep["ties"]["risk_index"] = int((idx_bad & ~real).sum())
                if real.any():
                    rep["fail"].append(f"max_obst_risk_index mismatch on {int(real.sum())} pairs")
        for col, name, atol in ((0, "max_ego_risk_all", ATOL_CP), (1, "max_obst_risk_all", ATOL_CP),
                                (2, "max_ego_harm_all", ATOL_HARM), (3, "max_obst_harm_all", ATOL_HARM),
                                (4, "max_collision_probability_all", ATOL_CP), (5, "max_obst_harm_with_cp_all", ATOL_HARM)):
            bad = ~_close(summ[:, col], out[name], RTOL, atol) & ~hr_tie_pair.any(1)
            if name == "max_obst_harm_with_cp_all" and bad.any() and pair is None:
                mcp = out["hr_pair"]["max_collision_probability"]
                bad &= ~(np.abs(mcp - 0.01) < 1e-5).any(1)
            if name == "max_obst_harm_with_cp_all" and bad.any():
                # tolerate trajectories whose per-pair value was already classified as a tie
                mcp = out["hr_pair"]["max_collision_probability"]
                srt = np.sort(out["cp"], -1)
                arg_tie = ((srt[..., -1] - srt[..., -2]) < 1e-4 * np.maximum(srt[..., -1], 1e-30)) & (mcp > 0.009)
                bad &= ~((np.abs(mcp - 0.01) < 1e-5) | arg_tie).any(1)
            if bad.any():
                i = int(np.argmax(bad))
                rep["fail"].append(f"summary {name} mismatch at traj {i}: gpu {summ[i, col]!r} oracle {out[name][i]!r} "
                                   f"({int(bad.sum())})")
        tie_traj |= hr_tie_pair.any(1)

    # ---------------------------------------------------------------- BE
    if "be" in order:
        if pair is not None:
            g = pair[..., 9].astype(np.float64)
            bad = ~_close(g, out["be_rcd"], 1e-5, 1e-6) & ok_traj[:, None] & ~dce_tie_pair
            n_be = int(((out["be_rcd"] > 0) & ok_traj[:, None]).sum())
            rep["n_be_pairs"] = n_be
            rep["ties"]["be_bisect"] = int(bad.sum())
            big = bad & (np.abs(g - out["be_rcd"]) > 2.6)
            if big.any():
                rep["fail"].append(f"BE mismatch larger than one bisection level on {int(big.sum())} pairs")
            tie_traj |= bad.any(1)
            gb = pair[..., 10].astype(np.float64)
            bad2 = ~_close(gb, out["be_btn"], 1e-5, 1e-6) & ok_traj[:, None] & ~bad & ~dce_tie_pair
            if bad2.any():
                rep["fail"].append(f"break_threat_number mismatch on {int(bad2.sum())} pairs")

    # ---------------------------------------------------------------- validity mask
    g_valid = res["valid"].astype(bool)
    bad = (g_valid != out["valid"]) & ok_traj
    # threshold ties: value within rtol of its threshold
    thr = case["thresholds"]
    near_thr = np.zeros(N, dtype=bool)
    if "hr" in order:
        for key, name in (("harm", "max_obst_harm_with_cp_all"), ("risk", "max_obst_risk_all"),
                          ("cp", "max_collision_probability_all")):
            if thr.get(key) is not None:
                near_thr |= np.abs(out[name] - thr[key]) <= RTOL * abs(thr[key]) + 1e-7
    rep["ties"]["mask"] = int((bad & (tie_traj | near_thr)).sum())
    hard = bad & ~(tie_traj | near_thr)
    rep["mask_mismatch"] = int(hard.sum())
    if hard.any():
        rep["fail"].append(f"validity mask differs on {int(hard.sum())} trajectories, first {int(np.argmax(hard))}")
    rep["n_valid"] = int(out["valid"].sum())
    return rep


def risk_index_tie(out, gpu_index):
    """Risk argmax tie, [...] like ``gpu_index`` (the kernel's max_obst_risk_index per pair): the oracle's obstacle
    risk at the kernel's index equals its maximum within rounding (1e-5 relative, 1e-12 absolute).  Either two float32
    risk products are equal within rounding, or all risks of the pair are below 1e-12 -- e.g. exact zeros where the
    float64 ndtr(hi) - ndtr(lo) of an interval more than ~8 sigma away cancels, while the kernels' erfc of the tails
    keeps a value of 1e-24, so the first maximum moves from step 0 to that step."""
    orr = np.nan_to_num(out["obst_risk"], nan=-1.0)
    v_g = np.take_along_axis(orr, gpu_index[..., None], -1)[..., 0]
    return _close(v_g, orr.max(-1), 1e-5, 1e-12)


def run_gpu(case, want_pair=True, want_step=True, device="cuda:0"):
    import torch
    from frenetix_occlusion_b200.engine import AgentSet, MetricEngine
    eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"], device=device)
    eng.set_agents(AgentSet.from_case(case["agents"]))
    r = eng.assess(np.asarray(case["ego"]), want_pair=want_pair, want_step=want_step)
    torch.cuda.synchronize()
    res = {"valid": r.valid.cpu().numpy(), "summary": r.summary.cpu().numpy(),
           "flags": r.flags.cpu().numpy().astype(np.uint32)}
    res["pair"] = r.pair.cpu().numpy() if r.pair is not None else None
    res["step"] = r.step.cpu().numpy() if r.step is not None else None
    return res, eng
