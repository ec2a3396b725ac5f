"""Assessment of several independent planning problems in one launch of the dense metric core.

A multi-agent simulation runs one planner and one ``FOInterface`` per vehicle; a re-simulation or parameter sweep runs
many scenes side by side.  Instead of one ``assess_bundle`` per interface (an agent upload, two pack launches and a
metric launch each), ``assess_interfaces`` packs the phantom agents of all interfaces with one
``fo_agents_pack_batch`` call and evaluates all candidate bundles with one ``fo_metric_batch`` (or, with pair / step
detail, ``fo_metric_batch_detail``) call -- their ``_corr`` forms when some interface's predictions carry correlated
covariances, which are then assessed as that interface assesses them.  ``prefetch_interfaces`` does the same for the reference's per-trajectory
protocol: it is ``prefetch_assessments`` for all interfaces at once, and ``select_interfaces`` gives each interface the
first candidate that passes, as ``FOInterface.select_trajectory`` does.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from . import _lib as L
from .engine import AgentSet, BatchResult, BundleResult, MetricEngine


def _config(fi) -> dict:
    """What the batched call shares across problems, read from an interface's metric engine."""
    eng = fi.metrics._core.engine
    h = eng.harm
    return {"device": torch.device(eng.device), "dt": eng.dt,
            "metrics": eng.metric_mask,
            "thresholds": (eng.threshold_mask, tuple(sorted(eng.thresholds.items(), key=lambda kv: kv[0]))),
            "harm": tuple(getattr(h, f) for f, _ in h._fields_)}


def _bundle_array(bundle):
    """A bundle as ``FOInterface.assess_bundle`` takes it: [N, T, 5] array / tensor or a sequence of trajectories."""
    if isinstance(bundle, (np.ndarray, torch.Tensor)):
        return bundle
    from .metrics.core import trajectory_to_array
    return np.stack([trajectory_to_array(t) for t in bundle])


def _batch_engine(interfaces, egos) -> MetricEngine:
    """An engine with the configuration the interfaces share (the ego vehicle is per problem: ``_vehicles``);
    ``ValueError`` when they or their trajectory lengths differ."""
    cfgs = [_config(fi) for fi in interfaces]
    for i, c in enumerate(cfgs[1:], 1):
        diff = [k for k in c if c[k] != cfgs[0][k]]
        if diff:
            raise ValueError(f"interface {i} differs from interface 0 in {', '.join(diff)}: one batch shares them")
    lengths = {int(e.shape[-2]) for e in egos if e.shape[0] > 0}
    if len(lengths) > 1:
        raise ValueError(f"trajectory lengths differ across interfaces: {sorted(lengths)}")
    eng0 = interfaces[0].metrics._core.engine
    return MetricEngine(eng0.vehicle, eng0.dt, list(eng0.order), eng0.thresholds,
                        harm_coeffs={f: getattr(eng0.harm, f) for f, _ in eng0.harm._fields_}, device=eng0.device)


def _vehicles(interfaces) -> list:
    """Each interface's ego vehicle, as its own metric engine holds it (from the interface's ``vehicle_params``)."""
    return [fi.metrics._core.engine.vehicle for fi in interfaces]


def _agents(fi):
    """An interface's phantom predictions and their origin, by the rule of ``MetricCore.sync_agents`` (the first
    agent's first position); none for an interface without phantom agents or metrics."""
    am = fi.agent_manager
    if am.phantom_agents and fi.metrics.metrics:
        ag = AgentSet.from_predictions(am.predictions, am.agent_by_prediction_id)
    else:
        ag = AgentSet.from_case([])
    return ag, ((float(ag.x[0, 0]), float(ag.y[0, 0])) if ag.n_agents else (0.0, 0.0))


def assess_interfaces(interfaces: Sequence, bundles: Sequence, want_pair: bool = False, want_step: bool = False) -> list:
    """Assess the candidate ``bundles[i]`` of every ``interfaces[i]`` (each after its ``evaluate_scenario`` of the
    current step) with one pack and one metric call for all of them.  Returns one ``engine.BundleResult`` per
    interface, views of shared device tensors, equal to what ``interfaces[i].assess_bundle(bundles[i], want_pair,
    want_step)`` gives.

    Each interface's phantom predictions (``agent_manager.predictions``) are taken with the origin rule of
    ``MetricCore.sync_agents`` (the first agent's first position); an interface without phantom agents assesses
    every trajectory as valid (``Metric.evaluate_metrics``).  Each interface is assessed with its own ego vehicle
    (``vehicle_params``), so the vehicles of a mixed fleet share one batch, and with its own predictions' covariances,
    diagonal or correlated.  The interfaces must agree on device, dt,
    activated metrics, thresholds, harm coefficients and the trajectory length T, else ``ValueError``.  No interface's
    state, cache or prefetch is touched."""
    interfaces, bundles = list(interfaces), list(bundles)
    if len(interfaces) != len(bundles):
        raise ValueError(f"{len(interfaces)} interfaces but {len(bundles)} bundles")
    if not interfaces:
        return []
    egos = [_bundle_array(b) for b in bundles]
    eng = _batch_engine(interfaces, egos)
    agents = [_agents(fi) for fi in interfaces]
    eng.set_agent_batch([a for a, _ in agents], [o for _, o in agents], vehicles=_vehicles(interfaces), correlated=True)
    return eng.assess_batch(egos, want_pair=want_pair, want_step=want_step).split()


def prefetch_interfaces(interfaces: Sequence, candidates: Sequence) -> list:
    """``interfaces[i].prefetch_assessments(candidates[i])`` for every interface at once: one ``fo_agents_pack_batch``,
    one ``fo_metric_batch_detail`` and one device-to-host copy of all results (with correlated predictions the ``_corr``
    calls: a third pack launch, and one detail launch each for the diagonal and the correlated interfaces).  Afterwards
    ``interfaces[i].trajectory_safety_assessment(t)`` for every ``t`` in ``candidates[i]`` (trajectory objects with
    ``.cartesian.x / y / theta / v / a``) returns what it would after the interface's own prefetch, without a launch.
    Returns the per-interface counts ``prefetch_assessments`` returns (0 for an interface without phantom agents or
    metrics, which is left untouched).  The configuration rule and ``ValueError`` are those of
    ``assess_interfaces``."""
    from .metrics.core import trajectory_to_array
    interfaces, candidates = list(interfaces), [list(c) for c in candidates]
    if len(interfaces) != len(candidates):
        raise ValueError(f"{len(interfaces)} interfaces but {len(candidates)} candidate lists")
    live = [i for i, fi in enumerate(interfaces) if fi.agent_manager.phantom_agents and fi.metrics.metrics]
    egos = [np.stack([trajectory_to_array(t) for t in candidates[i]]) if candidates[i] else np.zeros((0, 1, 5))
            for i in live]
    if not interfaces:
        return []
    eng = _batch_engine(interfaces, egos)
    counts = [0] * len(interfaces)
    if not live:
        return counts
    agents = [_agents(interfaces[i]) for i in live]
    eng.set_agent_batch([a for a, _ in agents], [o for _, o in agents],
                        vehicles=_vehicles([interfaces[i] for i in live]), correlated=True)
    n = np.array([len(e) for e in egos], dtype=np.int64)
    a = np.array([ag.n_agents if ag.t_stride > 0 else 0 for ag, _ in agents], dtype=np.int64)
    T = max([e.shape[1] for e in egos if len(e)], default=1)
    N, n_pairs, tm1 = int(n.sum()), int(np.dot(n, a)), T - 1
    # every output in one device buffer (one copy back), each part 16-byte aligned
    sizes = [N, 4 * N, 4 * N * L.FO_SUMMARY_K, 4 * n_pairs * L.FO_PAIR_K, 4 * n_pairs * tm1 * L.FO_STEP_K]
    offs = np.concatenate([[0], np.cumsum([(b + 15) // 16 * 16 for b in sizes])])
    dev = eng.device
    buf = torch.empty(max(int(offs[-1]), 16), dtype=torch.uint8, device=dev)
    part = lambda j: buf[int(offs[j]):int(offs[j]) + sizes[j]]  # noqa: E731
    out = BatchResult(part(0), part(2).view(torch.float32).view(N, L.FO_SUMMARY_K), part(1).view(torch.int32), None,
                      pair=part(3).view(torch.float32), step=part(4).view(torch.float32))
    with torch.cuda.device(dev):
        eng.assess_batch(egos, want_pair=True, want_step=True, out=out)
        host = buf.cpu().numpy()                     # synchronises the stream
    f32 = lambda j: host[int(offs[j]):int(offs[j]) + sizes[j]].view(np.float32).astype(np.float64)  # noqa: E731
    valid, flags = host[:N], host[int(offs[1]):int(offs[1]) + sizes[1]].view(np.uint32)
    summary, pair, step = f32(2).reshape(N, L.FO_SUMMARY_K), f32(3), f32(4)
    r, q = 0, 0
    for j, i in enumerate(live):
        nj, aj = int(n[j]), int(a[j])
        h = {"valid": valid[r:r + nj], "flags": flags[r:r + nj], "summary": summary[r:r + nj],
             "pair": pair[q * L.FO_PAIR_K:(q + nj * aj) * L.FO_PAIR_K].reshape(nj, aj, L.FO_PAIR_K),
             "step": step[q * tm1 * L.FO_STEP_K:(q + nj * aj) * tm1 * L.FO_STEP_K].reshape(nj, aj, tm1, L.FO_STEP_K),
             "ego": egos[j]}
        ag, origin = agents[j]
        counts[i] = interfaces[i].metrics._core.install_prefetch(candidates[i], h, agents=ag, origin=origin)
        r, q = r + nj, q + nj * aj
    return counts


def select_interfaces(interfaces: Sequence, candidates: Sequence) -> list:
    """``interfaces[i].select_trajectory(candidates[i])`` for every interface in one pack and one
    ``fo_metric_batch_select`` call: per interface the index of the first candidate (in the order given, the planner's
    cost order) that passes, or None when none does.  Configuration rule, vehicles, covariances and ``ValueError`` as in
    ``assess_interfaces``; an interface without phantom agents or metrics gets 0 (None for no candidates).  Synchronises
    on one int per interface; no interface's state, cache or prefetch is touched."""
    interfaces, candidates = list(interfaces), list(candidates)
    if len(interfaces) != len(candidates):
        raise ValueError(f"{len(interfaces)} interfaces but {len(candidates)} candidate lists")
    if not interfaces:
        return []
    egos = [_bundle_array(c) if len(c) else np.zeros((0, 1, 5)) for c in candidates]
    eng = _batch_engine(interfaces, egos)
    agents = [_agents(fi) for fi in interfaces]
    eng.set_agent_batch([a for a, _ in agents], [o for _, o in agents], vehicles=_vehicles(interfaces), correlated=True)
    r = eng.select_batch(egos)
    sel = r.selected.cpu().numpy()
    return [int(k) if k < n else None for k, n in zip(sel, np.diff(r.offsets))]


__all__ = ["assess_interfaces", "prefetch_interfaces", "select_interfaces", "BundleResult"]
