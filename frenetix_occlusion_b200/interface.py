"""Entry point of the assessment hot path (mirror of reference frenetix_occlusion/interface.py:18-238).

Same constructor, attributes and the three calls the planner makes -- ``evaluate_scenario`` once per planning
cycle, ``trajectory_safety_assessment`` per candidate trajectory -- plus the batched
``assess_bundle(trajectories[N,T,5])`` that evaluates the planner's whole sampled bundle in one launch of the
dense CUDA core (the call a planner should prefer; the per-trajectory call is one 1-trajectory launch).

Differences from the reference, all at its edges: ``config_path=None`` loads the package default instead of
crashing (interface.py:231-236 opens an unbound name); the debug visualisation is optional and never forces a
matplotlib backend; ``evaluate_scenario`` returns the visible area as a region object over the ray-cast map
instead of a shapely polygon."""
from __future__ import annotations

import os

import yaml

from .agent import FOAgentManager
from .metrics.metric import Metric
from .sensor_model import SensorModel
from .spawn_locator import SpawnLocator
from .utils.fo_obstacle import FOObstacles


class FOInterface:
    def __init__(self, scenario, reference_path, vehicle_params, dt, config_path=None, cosy_cl=None, device="cuda:0",
                 visualization=None, warm_up=True):
        self.config = self._load_config(config_path)
        self.cr_scenario = scenario
        self.lanelet_network = scenario.lanelet_network
        self.ego_reference_path = reference_path
        self.cosy_cl = cosy_cl
        self.vehicle_params = vehicle_params
        self.dt = dt
        self.plot = self.config["plot"]
        self.debug = self.config["debug"]
        self.device = device

        self.predictions = None
        self.ego_pos = None
        self.ego_orientation = None
        self.ego_pos_cl = None
        self.timestep = None
        self.spawn_points = []

        self.sensor_radius = self.config["sensor_model"]["sensor_radius"]
        self.sensor_angle = self.config["sensor_model"]["sensor_angle"]

        # the reference constructs its matplotlib visualisation unconditionally (interface.py:97); here it is an
        # optional object with the same drawing methods
        self.visualization = visualization

        self.fo_obstacles = FOObstacles(self.cr_scenario.obstacles)
        self.sensor_model = self._make_sensor_model()
        self.agent_manager = self._make_agent_manager()
        self.spawn_locator = SpawnLocator(agent_manager=self.agent_manager, ref_path=self.ego_reference_path,
                                          config=self.config, cosy_cl=self.cosy_cl, sensor_model=self.sensor_model,
                                          fo_obstacles=self.fo_obstacles, visualization=self.visualization,
                                          debug=self.debug)
        self.metrics = self._make_metrics()
        if warm_up:
            self._warm_up()

    # construction hooks (one per device-backed component)
    def _make_sensor_model(self):
        return SensorModel(lanelet_network=self.lanelet_network, ref_path=self.ego_reference_path,
                           sensor_radius=self.sensor_radius, sensor_angle=self.sensor_angle,
                           visualization=self.visualization, debug=self.debug, device=self.device)

    def _make_agent_manager(self):
        return FOAgentManager(scenario=self.cr_scenario, reference_path=self.ego_reference_path,
                              config=self.config["agent_manager"], visualization=self.visualization,
                              timestep=self.timestep, dt=self.dt, debug=self.debug, fo_obstacles=self.fo_obstacles,
                              device=self.device)

    def _make_metrics(self):
        return Metric(self.config["metrics"], self.vehicle_params, self.agent_manager, device=self.device)

    def _warm_up(self):
        """Pay the first-use costs (CUDA context, module load, page-locked staging buffers, kernel attributes) at
        construction instead of in the first planning cycle: one tiny call of every device entry point."""
        import numpy as np
        import scipy.ndimage  # noqa: F401  (the spawn locator's first use would otherwise pay the import in cycle 0)
        import scipy.spatial  # noqa: F401  (convex hull of the candidate-box outlines)
        import torch
        from .engine import AgentSet
        from .prediction import rollout_cv, rollout_path
        from .visibility import FrameGeometry
        if not torch.cuda.is_available() or not hasattr(self.sensor_model, "n_rays"):
            return
        road = [np.array([[-1.0, -2.0], [30.0, -2.0], [30.0, 4.0], [-1.0, 4.0]])]
        fr = FrameGeometry([0.0, 0.0], 0.0, np.array([[8.0, 0.5, 0.1, 2.0, 1.0]]), np.array([1], dtype=np.uint8),
                           np.array([[0.0, 4.0, 30.0, 4.0]]), road, self.sensor_radius, self.sensor_angle, device=self.device)
        fr.raycast_host(self.sensor_model.n_rays, road_hits=(0.0, 2.0 * np.pi / self.sensor_model.n_rays))
        fr.classify(np.array([[3.0, 1.0], [15.0, 0.5]]), focus_obstacle=0, focus_margin=1.0)
        # the device rasters of the dynamic-obstacle finder at the size a cycle uses: their workspace (the first
        # torch.zeros on a device loads torch's own kernel module: 0.5 s), page-locked result buffers, kernel modules
        from . import _lib as L
        half, cell = self.spawn_locator.buffer_around_vehicle_from_side, self.spawn_locator.raster_cell
        _, _, _, _, handle = fr.spawn_region(np.array([8.0, 0.5]), half, cell, int(np.ceil(2 * half / cell)), 1, L.PT_OCCLUDED,
                                             L.PT_FOCUS_NEAR, half, np.array([14.0, 0.5]), 0, 1.0)
        fr.spawn_rects(handle, [(np.array([14.0, 0.5]), 5.5, 2.5, False), (np.array([14.0, 0.5]), 2.0, 1.0, True)], 0.0,
                       self.spawn_locator.rect_cell)
        rollout_cv([1.0], [1.0], [1.4], [0.3], self.dt, 3.0, device=self.device)
        rollout_path([np.array([[0.0, 0.0], [20.0, 0.0], [40.0, 1.0]])], [2.0], [0.2], [5.0], self.dt, 3.0, device=self.device)
        core = getattr(self.metrics, "_core", None)
        if core is not None:
            n = int(round(3.0 / self.dt)) + 1
            t = np.arange(n) * self.dt
            agent = {"agent_type": "Pedestrian", "length": 0.3, "width": 0.5, "buf_length": 0.36, "buf_width": 0.65,
                     "pos": np.stack((12.0 + 0 * t, -3.0 + 1.4 * t), -1), "yaw": np.full(n, 1.57), "v": np.full(n, 1.4),
                     "var": 0.1 * 1.05 ** np.arange(n)}
            ego = np.stack((8.0 * t, 0 * t, 0 * t, 8.0 + 0 * t, 0 * t), -1)[None]
            core.engine.set_agents(AgentSet.from_case([agent]))
            core.engine.assess(ego)                                       # summary kernel
            core.engine.assess(ego, want_pair=True, want_step=True)       # detail kernel
            core.engine.set_agents(AgentSet.from_case([]))
            core._fingerprint = None
        torch.cuda.current_stream(torch.device(self.device)).synchronize()

    def set_coordinate_system(self, cosy_cl):
        self.cosy_cl = cosy_cl
        self.spawn_locator.cosy_cl = cosy_cl

    def _add_real_agents(self):
        """interface.py:137-146: configured real agents enter the scenario at their own time step."""
        if self.config["agents"] is None:
            return
        for agent in self.config["agents"]:
            self.agent_manager.add_agent(pos=agent["position"], velocity=agent["velocity"], agent_type=agent["agent_type"],
                                         add_to_scenario=True, timestep=agent["timestep"], horizon=agent["horizon"])

    def evaluate_scenario(self, predictions, ego_pos, ego_orientation, ego_pos_cl, ego_v, timestep, cosy_cl):
        """interface.py:148-214: visibility -> spawn points -> phantom agents (+ their predictions)."""
        self.set_coordinate_system(cosy_cl)
        self._update_time_step(timestep)
        self._add_real_agents()
        self.predictions = predictions
        self.ego_pos = ego_pos
        self.ego_orientation = ego_orientation
        self.ego_pos_cl = ego_pos_cl
        self.agent_manager.reset()
        self.spawn_points.clear()
        if self.visualization is not None and self.plot:
            self.visualization.draw_scenario(timestep=self.timestep)
            self.visualization.show_plot()
        self.fo_obstacles.update(self.timestep)
        self.sensor_model.calc_visible_and_occluded_area(timestep=self.timestep, ego_pos=self.ego_pos,
                                                         ego_orientation=self.ego_orientation, obstacles=self.fo_obstacles)
        self.fo_obstacles.update_multipolygon()
        self.spawn_points = self.spawn_locator.find_spawn_points(self.ego_pos, self.ego_orientation, self.ego_pos_cl, ego_v)
        # interface.py:187-198, all phantom agents of the cycle rolled out in one device pass
        self.agent_manager.add_agents([
            dict(pos=sp.position, velocity="default", agent_type=sp.agent_type, timestep=self.timestep, horizon=3.0,
                 mode="lane_center" if sp.source == "left turn" or sp.source == "right turn" else "ref_path",
                 orientation=sp.orientation) for sp in self.spawn_points])
        if self.debug:
            for sp, agent in zip(self.spawn_points, self.agent_manager.phantom_agents):
                print("Phantom agent of type {} with id {} added to scenario at position {}"
                      .format(sp.agent_type, agent.agent_id, sp.position))
        self.agent_manager.update_real_agents(self.predictions)
        if self.visualization is not None and self.plot:
            self.visualization.draw_predictions(self.agent_manager.predictions, label=False)
            self.visualization.show_plot(time=0.1)
        return self.sensor_model.visible_area

    def trajectory_safety_assessment(self, trajectory):
        """interface.py:216-219."""
        metrics, safety_assessment = self.metrics.evaluate_metrics(trajectory)
        return metrics, safety_assessment

    def prefetch_assessments(self, trajectories):
        """Optional companion of the per-trajectory protocol: hand over the cycle's candidate objects once; their
        detailed results are computed in ONE launch and ``trajectory_safety_assessment`` then answers from the host
        copy (same dicts, about 20 us per call instead of a launch + blocking read-back each)."""
        return self.metrics.prefetch(trajectories)

    def assess_bundle(self, trajectories, want_pair=False, want_step=False):
        """Whole sampled bundle at once: ``trajectories`` is [N, T, 5] (x, y, theta, v, a) as a tensor / array or a
        sequence of trajectory objects.  Returns device tensors ``valid[N]``, ``summary[N, K]``, ``flags[N]``
        (``engine.BundleResult``); every trajectory is valid when there are no phantom agents (metric.py:44-45)."""
        return self.metrics.evaluate_bundle(trajectories, want_pair=want_pair, want_step=want_step)

    def select_trajectory(self, trajectories):
        """The planner's protocol in one call: ``trajectories`` sorted by cost (as ``assess_bundle`` takes them), the
        index of the first one ``trajectory_safety_assessment`` would pass, or None when none passes.  Only the
        candidates up to that one need to be assessed.  For the chosen candidate's result dict call
        ``trajectory_safety_assessment(trajectories[k])``; the prefetch is not touched."""
        return self.metrics.select(trajectories)

    def _update_time_step(self, timestep):
        self.timestep = timestep
        self.sensor_model.timestep = timestep
        self.agent_manager.timestep = timestep

    @staticmethod
    def _load_config(filepath: str = None):
        if isinstance(filepath, dict):          # extension: an already-parsed configuration
            import copy
            return copy.deepcopy(filepath)
        if not filepath:
            filepath = os.path.join(os.path.dirname(__file__), "config", "config.yaml")
            print("Load default occlusion module settings!")
        with open(filepath, "r") as file:
            return yaml.safe_load(file)
