"""Metric dispatcher (mirrors reference frenetix_occlusion/metrics/metric.py:18-147).

Same constructor, plugin registry, dependency ordering and threshold logic; the numbers come from
one launch of the CUDA dense core per trajectory (``evaluate_metrics``) or per bundle
(``evaluate_bundle``, the batched entry the planner should prefer)."""
from __future__ import annotations

from .be import BE
from .core import MetricCore
from .cp import CP
from .dce import DCE
from .hr import HR
from .ttc import TTC
from .ttce import TTCE
from .wttc import WTTC


class Metric:
    def __init__(self, config, vehicle_params, agent_manager, device="cuda:0"):
        self.config = config
        self.metric_thresholds = config["metric_thresholds"]
        self.vehicle_params = vehicle_params
        self.agent_manager = agent_manager
        names = self._check_required_metrics(self.config["activated_metrics"])
        # ONE source for the harm coefficients: the JSON the HR plugin loads (hr.py:20-24) also feeds the kernel
        from ..engine import harm_from_reference_json
        self._core = MetricCore(vehicle_params, agent_manager, activated_metrics=[n for n in names],
                                thresholds=self.metric_thresholds, device=device,
                                harm_coeffs=harm_from_reference_json(HR._load_param("harm_coefficients")))
        self.metrics = self._initialize_metrics(names)

    # ---- per trajectory (reference metric.py:35-100) ---------------------------------------------
    def evaluate_metrics(self, trajectory):
        results = {}
        if not self.agent_manager.phantom_agents or not self.metrics:
            return results, True
        self._core.begin(trajectory)             # the plugins of this call share one launch; nothing older is reused
        try:
            for name, metric in self.metrics.items():
                results[name] = metric.evaluate(trajectory, results)
        finally:
            self._core.end()

        thr = self.metric_thresholds
        safety_check = True
        if "be" in results and thr["be"] is not None:
            for key in results["be"]:
                if results["be"][key]["break_threat_number"] > thr["be"]:
                    safety_check = False
                    break
        if "hr" in results and thr["harm"] is not None:
            if results["hr"]["max_obst_harm_with_cp_all"] > thr["harm"]:
                safety_check = False
        if "hr" in results and thr["risk"] is not None:
            if results["hr"]["max_obst_risk_all"] > thr["risk"]:
                safety_check = False
        if "hr" in results and thr["cp"] is not None:
            if results["hr"]["max_collision_probability_all"] > thr["cp"]:
                safety_check = False
        if "ttc" in results and thr["ttc"] is not None:
            if min(results["ttc"].values()) < thr["ttc"]:
                safety_check = False
        if "dce" in results and thr["dce"] is not None:
            for key in results["dce"]:
                if results["dce"][key]["dce"] < thr["dce"]:
                    safety_check = False
                    break
        return results, safety_check

    # ---- whole bundle (new, batched) ---------------------------------------------------------------
    def evaluate_bundle(self, trajectories, want_pair=False, want_step=False):
        """``trajectories``: [N, T, 5] tensor/array (x, y, theta, v, a) or a sequence of trajectory
        objects.  Returns ``engine.BundleResult`` (device tensors: valid[N], summary[N, K], flags[N])."""
        import numpy as np
        import torch
        from .core import trajectory_to_array
        if not isinstance(trajectories, (np.ndarray, torch.Tensor)):
            trajectories = np.stack([trajectory_to_array(t) for t in trajectories])
        return self._core.bundle(trajectories, want_pair=want_pair, want_step=want_step)

    def select(self, trajectories):
        """Index of the first of ``trajectories`` (in priority order: [N, T, 5] tensor / array or a sequence of
        trajectory objects) that ``evaluate_metrics`` finds safe, None when none is; 0 without phantom agents or
        metrics (metric.py:44-45), None for an empty list.  Only the rows up to the answer need to be assessed
        (``MetricEngine.select``); synchronises on one int, and leaves the prefetch untouched."""
        import numpy as np
        import torch
        from .core import trajectory_to_array
        if not isinstance(trajectories, (np.ndarray, torch.Tensor)):
            trajectories = list(trajectories)
            if not trajectories:
                return None
            trajectories = np.stack([trajectory_to_array(t) for t in trajectories])
        if int(trajectories.shape[0]) == 0:
            return None
        if not self.agent_manager.phantom_agents or not self.metrics:
            return 0
        return self._core.select(trajectories)

    def prefetch(self, trajectories):
        """Evaluate all candidates of this planning cycle in one launch; the ``evaluate_metrics`` calls that follow are
        served from the host copy (see ``MetricCore.prefetch``)."""
        if not self.agent_manager.phantom_agents or not self.metrics:
            return 0
        return self._core.prefetch(trajectories)

    def register(self, name, metric, position=None):
        """Plug in a user metric: any object with ``evaluate(trajectory, results)``."""
        items = list(self.metrics.items())
        items.insert(len(items) if position is None else position, (name, metric))
        self.metrics = dict(items)

    def _initialize_metrics(self, metric_names):
        core = self._core
        metric_classes = {
            "dce": DCE(self.vehicle_params, self.agent_manager, core=core),
            "cp": CP(self.vehicle_params, self.agent_manager, core=core),
            "ttc": TTC(self.agent_manager),
            "ttce": TTCE(self.agent_manager),
            "wttc": WTTC,
            "be": BE(self.vehicle_params, self.agent_manager, core=core),
            "hr": HR(self.vehicle_params, self.agent_manager, core=core),
        }
        return {name: metric_classes[name] if type(metric_classes[name]) is not type else metric_classes[name]()
                for name in metric_names if name in metric_classes}

    @staticmethod
    def _check_required_metrics(metric_names):
        """Dependency ordering; like the reference (metric.py:125-147) it edits the list in place."""
        if "wttc" in metric_names:
            if "ttc" in metric_names:
                metric_names.remove("ttc")
            metric_names.insert(0, "ttc")
        if "ttc" in metric_names or "ttce" in metric_names or "be" in metric_names:
            if "dce" in metric_names:
                metric_names.remove("dce")
            metric_names.insert(0, "dce")
        if "hr" in metric_names:
            if "cp" in metric_names:
                metric_names.remove("cp")
            metric_names.insert(0, "cp")
        return metric_names
