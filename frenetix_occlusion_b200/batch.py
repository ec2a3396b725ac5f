"""Assessment of several independent planning problems in one launch of the dense metric core.

A multi-agent simulation runs one planner and one ``FOInterface`` per vehicle; a re-simulation or parameter sweep runs
many scenes side by side.  Instead of one ``assess_bundle`` per interface (an agent upload, two pack launches and a
metric launch each), ``assess_interfaces`` packs the phantom agents of all interfaces with one
``fo_agents_pack_batch`` call and evaluates all candidate bundles with one ``fo_metric_batch`` call.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from .engine import AgentSet, BundleResult, MetricEngine


def _config(fi) -> dict:
    """What the batched call shares across problems, read from an interface's metric engine."""
    eng = fi.metrics._core.engine
    v, h = eng.vehicle, eng.harm
    return {"device": torch.device(eng.device), "dt": eng.dt,
            "vehicle": tuple(getattr(v, f) for f, _ in v._fields_),
            "metrics": eng.metric_mask,
            "thresholds": (eng.threshold_mask, tuple(sorted(eng.thresholds.items(), key=lambda kv: kv[0]))),
            "harm": tuple(getattr(h, f) for f, _ in h._fields_)}


def _bundle_array(bundle):
    """A bundle as ``FOInterface.assess_bundle`` takes it: [N, T, 5] array / tensor or a sequence of trajectories."""
    if isinstance(bundle, (np.ndarray, torch.Tensor)):
        return bundle
    from .metrics.core import trajectory_to_array
    return np.stack([trajectory_to_array(t) for t in bundle])


def assess_interfaces(interfaces: Sequence, bundles: Sequence) -> list:
    """Assess the candidate ``bundles[i]`` of every ``interfaces[i]`` (each after its ``evaluate_scenario`` of the
    current step) with one pack and one metric call for all of them.  Returns one ``engine.BundleResult`` per
    interface, views of shared device tensors, equal to what ``interfaces[i].assess_bundle(bundles[i])`` gives.

    Each interface's phantom predictions (``agent_manager.predictions``) are taken with the origin rule of
    ``MetricCore.sync_agents`` (the first agent's first position); an interface without phantom agents assesses
    every trajectory as valid (``Metric.evaluate_metrics``).  The interfaces must agree on device, dt, vehicle
    parameters, activated metrics, thresholds, harm coefficients and the trajectory length T, else ``ValueError``.
    No interface's state, cache or prefetch is touched."""
    interfaces, bundles = list(interfaces), list(bundles)
    if len(interfaces) != len(bundles):
        raise ValueError(f"{len(interfaces)} interfaces but {len(bundles)} bundles")
    if not interfaces:
        return []
    cfgs = [_config(fi) for fi in interfaces]
    for i, c in enumerate(cfgs[1:], 1):
        diff = [k for k in c if c[k] != cfgs[0][k]]
        if diff:
            raise ValueError(f"interface {i} differs from interface 0 in {', '.join(diff)}: one batch shares them")
    egos = [_bundle_array(b) for b in bundles]
    lengths = {int(e.shape[-2]) for e in egos if e.shape[0] > 0}
    if len(lengths) > 1:
        raise ValueError(f"trajectory lengths differ across interfaces: {sorted(lengths)}")
    agent_sets, origins = [], []
    for fi in interfaces:
        am = fi.agent_manager
        if am.phantom_agents and fi.metrics.metrics:
            ag = AgentSet.from_predictions(am.predictions, am.agent_by_prediction_id)
        else:
            ag = AgentSet.from_case([])
        origins.append((float(ag.x[0, 0]), float(ag.y[0, 0])) if ag.n_agents else (0.0, 0.0))
        agent_sets.append(ag)
    eng0 = interfaces[0].metrics._core.engine
    eng = MetricEngine(dict(zip(("length", "width", "mass", "wb_rear_axle", "a_max"), cfgs[0]["vehicle"])), eng0.dt,
                       list(eng0.order), eng0.thresholds,
                       harm_coeffs={f: getattr(eng0.harm, f) for f, _ in eng0.harm._fields_}, device=eng0.device)
    eng.set_agent_batch(agent_sets, origins)
    return eng.assess_batch(egos).split()


__all__ = ["assess_interfaces", "BundleResult"]
