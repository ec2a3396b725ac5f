"""Shared device evaluation behind the metric plugins.

One ``MetricCore`` serves all plugin objects of a ``Metric``: the first plugin asked about a
trajectory triggers ONE launch of the dense kernel (pair + step detail for a 1-trajectory bundle),
the others read the cached device results.  Agents are re-packed whenever the agent manager's
``predictions`` change (new planning cycle).
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib as L
from ..engine import AgentSet, BundleResult, MetricEngine

_ALL = ["hr", "ttc", "be", "ttce", "dce", "wttc", "cp"]


def trajectory_to_array(trajectory) -> np.ndarray:
    """``trajectory.cartesian.{x,y,theta,v,a}`` -> float64 [T, 5] (SURVEY.md 8b duck type)."""
    c = trajectory.cartesian
    return np.stack([np.asarray(c.x, dtype=np.float64), np.asarray(c.y, dtype=np.float64),
                     np.asarray(c.theta, dtype=np.float64), np.asarray(c.v, dtype=np.float64),
                     np.asarray(c.a, dtype=np.float64)], axis=-1)


class MetricCore:
    def __init__(self, vehicle_params, agent_manager, activated_metrics=None, thresholds=None, harm_coeffs=None,
                 device="cuda:0"):
        self.agent_manager = agent_manager
        self.vehicle_params = vehicle_params
        thresholds = thresholds or {}
        self.engine = MetricEngine(vehicle_params, agent_manager.dt, list(activated_metrics or _ALL), thresholds,
                                   harm_coeffs=harm_coeffs, device=device)
        self._fingerprint = None
        # result cache of ONE trajectory.  Two ways to hit it, neither relies on id() of an object that may have been
        # freed: (a) identity with the trajectory pinned by ``begin`` (a strong reference held for the duration of
        # one Metric.evaluate_metrics call), (b) equal contents (the stacked [T, 5] array is compared).
        self._pinned = None
        self._cache = None
        self._cache_ego = None
        # results of a whole bundle evaluated ahead of the per-trajectory calls (``prefetch``): id -> (trajectory, row)
        self._prefetched = {}
        self._prefetch_host = None

    # ---- agents --------------------------------------------------------------------------------
    def _agents_fingerprint(self):
        preds = self.agent_manager.predictions
        ver = getattr(self.agent_manager, "version", None)
        if ver is not None:                      # the product's FOAgentManager counts its modifications
            return ("v", ver, len(preds))
        # foreign managers (the reference's own FOAgentManager has no counter): fingerprint the contents
        items = []
        for k, v in preds.items():
            pos = np.ascontiguousarray(v.get("pos_list"), dtype=np.float64)
            items.append((k, pos.shape, hash(pos.tobytes()),
                          hash(np.ascontiguousarray(v.get("orientation_list"), dtype=np.float64).tobytes()),
                          hash(np.ascontiguousarray(v.get("v_list"), dtype=np.float64).tobytes()),
                          hash(np.ascontiguousarray(v.get("cov_list"), dtype=np.float64).tobytes())))
        return ("c", tuple(items))

    def sync_agents(self, origin=None):
        fp = self._agents_fingerprint()
        if fp == self._fingerprint:
            return
        preds = self.agent_manager.predictions
        agents = AgentSet.from_predictions(preds, self.agent_manager.agent_by_prediction_id)
        if origin is None and agents.n_agents:
            origin = (float(agents.x[0, 0]), float(agents.y[0, 0]))
        self.engine.set_agents(agents, origin=origin)
        self._fingerprint = fp
        self._cache = self._cache_ego = None
        self._prefetched = {}
        self._prefetch_host = None

    # ---- one evaluate_metrics call ------------------------------------------------------------------------
    def begin(self, trajectory):
        """Start of one ``Metric.evaluate_metrics(trajectory)``: re-check the agents once and pin the trajectory so
        that the plugins of this call share one launch."""
        self.sync_agents()
        self._pinned = trajectory
        self._cache = self._cache_ego = None

    def end(self):
        self._pinned = None

    # ---- whole candidate list ahead of the per-trajectory protocol ----------------------------------------------
    def prefetch(self, trajectories):
        """Evaluate every candidate of a planning cycle with full detail in ONE launch and ONE device-to-host copy;
        the per-trajectory calls that follow (reference protocol, interface.py:216-219) are served from the host
        copy.  The trajectory objects are held (strong references) until the agents change or the next prefetch."""
        self.sync_agents()
        trajectories = list(trajectories)
        self._prefetched, self._prefetch_host = {}, None
        if not trajectories:
            return 0
        ego = np.stack([trajectory_to_array(t) for t in trajectories])
        r = self.engine.assess(ego, want_pair=True, want_step=True)
        host = {"valid": r.valid.cpu().numpy(), "flags": r.flags.cpu().numpy().astype(np.uint32),
                "summary": r.summary.cpu().numpy().astype(np.float64),
                "pair": r.pair.cpu().numpy().astype(np.float64), "step": r.step.cpu().numpy().astype(np.float64),
                "ego": ego}
        return self.install_prefetch(trajectories, host)

    def install_prefetch(self, trajectories, host, agents=None, origin=None):
        """Serve the per-trajectory calls for ``trajectories`` (row k of ``host`` belongs to ``trajectories[k]``) from
        the host results ``host``: valid [N], flags [N], summary [N, K], pair [N, A, FO_PAIR_K], step [N, A, T-1,
        FO_STEP_K] and the stacked ego [N, T, 5].  ``agents`` / ``origin``: the agent set the results were computed for,
        when they were computed outside this core (``batch.prefetch_interfaces``).  It becomes the core's agent set for
        the current predictions without a pack of its own; a trajectory that misses the prefetch packs it first."""
        if agents is not None:
            self.engine._adopt_agents(agents, origin=origin)
            self._fingerprint = self._agents_fingerprint()
            self._cache = self._cache_ego = None
        self._prefetch_host = host if trajectories else None
        self._prefetched = {id(t): (t, k) for k, t in enumerate(trajectories)}
        return len(trajectories)

    def _from_prefetch(self, trajectory, ego):
        hit = self._prefetched.get(id(trajectory))
        if hit is None or hit[0] is not trajectory:
            return None
        h, k = self._prefetch_host, hit[1]
        if h["ego"][k].shape != ego.shape or not np.array_equal(h["ego"][k], ego):
            return None                           # mutated in place since the prefetch
        ag = self.engine.agents
        return {"valid": bool(h["valid"][k]), "flags": int(h["flags"][k]), "summary": h["summary"][k],
                "pair": h["pair"][k], "step": h["step"][k], "ids": list(ag.ids) if ag is not None else [],
                "n_states": ag.n_states if ag is not None else np.zeros(0, int), "T": ego.shape[0]}

    # ---- one trajectory, full detail --------------------------------------------------------------
    def detail(self, trajectory):
        if trajectory is self._pinned and self._cache is not None:
            return self._cache
        if trajectory is not self._pinned:
            self.sync_agents()
        ego = trajectory_to_array(trajectory)
        if self._cache is not None and self._cache_ego is not None and self._cache_ego.shape == ego.shape \
                and np.array_equal(self._cache_ego, ego):
            return self._cache
        if self._prefetched:
            d = self._from_prefetch(trajectory, ego)
            if d is not None:
                self._cache, self._cache_ego = d, ego
                return d
        A = self.engine.n_agents
        T = ego.shape[0]
        # all outputs of the 1-trajectory launch live in ONE device buffer -> one device-to-host copy
        n_pair, n_step = A * L.FO_PAIR_K, A * max(T - 1, 0) * L.FO_STEP_K
        off_flags, off_sum = 16, 32
        off_pair = off_sum + 4 * ((L.FO_SUMMARY_K + 3) // 4 * 4)
        off_step = off_pair + 4 * n_pair
        total = off_step + 4 * n_step
        dev = self.engine.device
        buf = torch.empty(max(total, 64), dtype=torch.uint8, device=dev)
        out = BundleResult(buf[0:1], buf[off_sum:off_sum + 4 * L.FO_SUMMARY_K].view(torch.float32).view(1, L.FO_SUMMARY_K),
                           buf[off_flags:off_flags + 4].view(torch.int32))
        out.pair = buf[off_pair:off_pair + 4 * n_pair].view(torch.float32).view(1, A, L.FO_PAIR_K)
        out.step = buf[off_step:off_step + 4 * n_step].view(torch.float32).view(1, A, max(T - 1, 0), L.FO_STEP_K)
        self.engine.assess(ego[None], out=out)
        host = buf.cpu().numpy()          # synchronises the stream
        f32 = lambda lo, n: host[lo:lo + 4 * n].view(np.float32).astype(np.float64)  # noqa: E731
        d = {"valid": bool(host[0]), "flags": int(host[off_flags:off_flags + 4].view(np.uint32)[0]),
             "summary": f32(off_sum, L.FO_SUMMARY_K),
             "pair": f32(off_pair, n_pair).reshape(A, L.FO_PAIR_K) if A else np.zeros((0, L.FO_PAIR_K)),
             "step": f32(off_step, n_step).reshape(A, T - 1, L.FO_STEP_K) if (A and T > 1) else np.zeros((A, 0, L.FO_STEP_K)),
             "ids": list(self.engine.agents.ids) if self.engine.agents is not None else [],
             "n_states": self.engine.agents.n_states if self.engine.agents is not None else np.zeros(0, int),
             "T": T}
        self._cache, self._cache_ego = d, ego
        return d

    # ---- a whole bundle, masks + summaries only ------------------------------------------------------
    def bundle(self, ego, want_pair=False, want_step=False):
        self.sync_agents()
        return self.engine.assess(ego, want_pair=want_pair, want_step=want_step)

    # ---- the first valid row of a bundle in priority order --------------------------------------------
    def select(self, ego):
        """Index of the first valid row of ``ego`` (``MetricEngine.select``), None when no row is valid; synchronises
        on one int.  The prefetch and the per-trajectory cache are left as they are."""
        self.sync_agents()
        n = int(ego.shape[0])
        k = int(self.engine.select(ego).selected.item())
        return k if k < n else None


_cores = {}


def shared_core(vehicle_params, agent_manager) -> MetricCore:
    """Core used by plugin objects constructed stand-alone (all seven metrics enabled)."""
    key = (id(vehicle_params), id(agent_manager))
    core = _cores.get(key)
    if core is None or core.agent_manager is not agent_manager or core.vehicle_params is not vehicle_params:
        core = MetricCore(vehicle_params, agent_manager)
        _cores.clear()
        _cores[key] = core
    return core
