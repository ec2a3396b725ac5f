"""Host side of the dense metric core: packs phantom-agent predictions and trajectory bundles into
device tensors and calls the sm_100a kernels through the C ABI (``include/fo_b200.h``).

PyTorch is used for device memory, streams and (in ``parallel.py``) ``torch.distributed`` only; all
arithmetic of the path happens in ``libfo_b200.so``.  No CPU fallback exists.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib as L

# harm coefficients read on this path; same keys/values as the reference's
# frenetix_occlusion/config/harm_params.json (log_reg.reduced_sym_angle_areas, log_reg.ignore_angle,
# pedestrian), see config/harm_coefficients.json
DEFAULT_HARM = {"rs_const": -4.457, "rs_speed": 0.177, "rs_side": 0.244, "rs_rear": -0.431,
                "ia_const": -4.591, "ia_speed": 0.185, "ped_const": 3.164, "ped_speed": 0.288}


def harm_from_reference_json(coeffs: dict) -> dict:
    """Map the reference's ``harm_params.json`` schema onto the kernel's coefficient block."""
    rs = coeffs["log_reg"]["reduced_sym_angle_areas"]
    ia = coeffs["log_reg"]["ignore_angle"]
    ped = coeffs["pedestrian"]
    return {"rs_const": rs["const"], "rs_speed": rs["speed"], "rs_side": rs["side"], "rs_rear": rs["rear"],
            "ia_const": ia["const"], "ia_speed": ia["speed"], "ped_const": ped["const"], "ped_speed": ped["speed"]}


def vehicle_struct(vehicle_params) -> L.FoVehicle:
    """An ego vehicle description (dict or object with attributes length, width, mass, wb_rear_axle, a_max) as the
    C ABI's ``FoVehicle``."""
    g = (lambda k: float(vehicle_params[k])) if isinstance(vehicle_params, dict) else \
        (lambda k: float(getattr(vehicle_params, k)))
    return L.FoVehicle(g("length"), g("width"), g("mass"), g("wb_rear_axle"), g("a_max"))


def check_required_metrics(metric_names: Sequence[str]) -> list:
    """Dependency ordering of the activated metrics (reference metrics/metric.py:125-147)."""
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
    return [x for x in m if x in L.M_BITS]


@dataclass
class AgentSet:
    """Phantom-agent predictions as padded SoA host arrays (what ``FOAgentManager.predictions`` holds,
    reference agent.py:420-424, 530-534, plus the owning agent's type / unbuffered shape)."""
    ids: list
    x: np.ndarray
    y: np.ndarray
    yaw: np.ndarray
    v: np.ndarray
    var_x: np.ndarray
    var_y: np.ndarray
    n_states: np.ndarray
    kind: np.ndarray
    length: np.ndarray
    width: np.ndarray
    buf_length: np.ndarray
    buf_width: np.ndarray
    agent_types: list = field(default_factory=list)
    # off-diagonal term of every covariance [A, t_stride], aligned with var_x / var_y; None = all diagonal
    cov_xy: Optional[np.ndarray] = None

    @property
    def n_agents(self) -> int:
        return len(self.ids)

    @property
    def t_stride(self) -> int:
        return int(self.x.shape[1]) if self.x.ndim == 2 else 0

    @staticmethod
    def _alloc(A, Tp):
        f = lambda: np.zeros((A, Tp), dtype=np.float64)  # noqa: E731
        return f(), f(), f(), f(), f(), f()

    @classmethod
    def from_case(cls, agents: Sequence[dict]) -> "AgentSet":
        """From the plain-array case format used by the tests / bench (see oracle/ref_runner.py)."""
        A = len(agents)
        Tp = max([len(np.asarray(a["yaw"])) for a in agents], default=0)
        x, y, yaw, v, vx, vy = cls._alloc(A, Tp)
        cxy = np.zeros((A, Tp), dtype=np.float64)
        ns = np.zeros(A, dtype=np.int32)
        kind = np.zeros(A, dtype=np.int32)
        dims = np.zeros((4, A), dtype=np.float64)
        types = []
        for k, a in enumerate(agents):
            n = len(np.asarray(a["yaw"]))
            ns[k] = n
            pos = np.asarray(a["pos"], dtype=np.float64).reshape(-1, 2)
            x[k, :n], y[k, :n] = pos[:, 0], pos[:, 1]
            yaw[k, :n], v[k, :n] = a["yaw"], a["v"]
            if "cov" in a:
                cov = np.asarray(a["cov"], dtype=np.float64)
                c01, c10, c00, c11 = cov[:, 0, 1], cov[:, 1, 0], cov[:, 0, 0], cov[:, 1, 1]
                if np.any(c01 != c10):
                    raise ValueError(f"agent {k}: prediction covariance is not symmetric")
                # positive definite where there is a correlation (scipy's mvn raises otherwise); diagonal states keep
                # the rules of the diagonal path (an all-zero matrix is 0.1 I)
                bad = (c01 != 0) & ~((c00 > 0) & (c11 > 0) & (c01 * c01 < c00 * c11))
                if np.any(bad):
                    raise ValueError(f"agent {k}: prediction covariance of state {int(np.argmax(bad))} is not positive definite")
                vx[k, :n], vy[k, :n], cxy[k, :n] = c00, c11, c01
            else:
                vx[k, :n] = vy[k, :n] = a["var"]
            kind[k] = L.KINDS[a["agent_type"].lower()]
            types.append(a["agent_type"])
            dims[:, k] = (a["length"], a["width"], a["buf_length"], a["buf_width"])
        return cls(list(range(A)), x, y, yaw, v, vx, vy, ns, kind, dims[0], dims[1], dims[2], dims[3], types,
                   cxy if np.any(cxy != 0) else None)

    @classmethod
    def from_predictions(cls, predictions: dict, agent_by_prediction_id) -> "AgentSet":
        """From the reference's own structures: ``agent_manager.predictions`` and
        ``agent_manager.agent_by_prediction_id`` (agent.py:159-183)."""
        agents = []
        ids = []
        for pid, pred in predictions.items():
            ag = agent_by_prediction_id(pid)
            cov = np.asarray(pred["cov_list"], dtype=np.float64)
            agents.append({"agent_type": ag.agent_type, "length": ag.shape.length, "width": ag.shape.width,
                           "buf_length": pred["shape"]["length"], "buf_width": pred["shape"]["width"],
                           "pos": pred["pos_list"], "yaw": pred["orientation_list"], "v": pred["v_list"],
                           "cov": cov})
            ids.append(pid)
        out = cls.from_case(agents)
        out.ids = ids
        return out


@dataclass
class BundleResult:
    valid: torch.Tensor                # uint8 [N]
    summary: torch.Tensor              # float32 [N, FO_SUMMARY_K]
    flags: torch.Tensor                # int32 [N]
    pair: Optional[torch.Tensor] = None   # float32 [N, A, FO_PAIR_K]
    step: Optional[torch.Tensor] = None   # float32 [N, A, T-1, FO_STEP_K]
    peer_delta: Optional[Sequence[int]] = None   # byte offsets to the peer-mapped copies of valid / summary / flags (parallel.py)


@dataclass
class BatchResult:
    """Results of a batch of independent problems: rows ``offsets[p]:offsets[p+1]`` belong to problem p.  The detail
    outputs are flat: problem p's [N_p, A_p, ...] blocks sit back to back in problem order (``fo_metric_batch_detail``)."""
    valid: torch.Tensor                # uint8 [N_total]
    summary: torch.Tensor              # float32 [N_total, FO_SUMMARY_K]
    flags: torch.Tensor                # int32 [N_total]
    offsets: np.ndarray                # int64 [P + 1]
    pair: Optional[torch.Tensor] = None     # float32 [sum_p N_p A_p FO_PAIR_K]
    step: Optional[torch.Tensor] = None     # float32 [sum_p N_p A_p (T-1) FO_STEP_K]
    n_agents: Optional[np.ndarray] = None   # A_p, with pair / step
    n_states: int = 0                       # T, with pair / step

    def split(self) -> list:
        """Per-problem ``BundleResult`` views of the batch tensors (no copies): pair [N_p, A_p, FO_PAIR_K] and step
        [N_p, A_p, T-1, FO_STEP_K] where the batch has them."""
        o = [int(x) for x in self.offsets]
        out, q, tm1 = [], 0, max(self.n_states - 1, 0)
        for p in range(len(o) - 1):
            r = BundleResult(self.valid[o[p]:o[p + 1]], self.summary[o[p]:o[p + 1]], self.flags[o[p]:o[p + 1]])
            n, a = o[p + 1] - o[p], int(self.n_agents[p]) if self.n_agents is not None else 0
            if self.pair is not None:
                r.pair = self.pair[q * L.FO_PAIR_K:(q + n * a) * L.FO_PAIR_K].view(n, a, L.FO_PAIR_K)
            if self.step is not None:
                r.step = self.step[q * tm1 * L.FO_STEP_K:(q + n * a) * tm1 * L.FO_STEP_K].view(n, a, tm1, L.FO_STEP_K)
            q += n * a
            out.append(r)
        return out


class MetricEngine:
    """Owns the device-side agent table and launches ``fo_metric_bundle``."""

    def __init__(self, vehicle_params, dt: float, activated_metrics: Sequence[str], thresholds: dict,
                 harm_coeffs: Optional[dict] = None, device="cuda:0"):
        if not torch.cuda.is_available():
            raise RuntimeError("frenetix_occlusion_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device)
        self.vehicle = vehicle_struct(vehicle_params)
        self.dt = float(dt)
        self.order = check_required_metrics(activated_metrics)
        if "be" in self.order and "ttc" not in self.order:
            raise KeyError("ttc")      # reference: be.py:39 reads results['ttc']
        self.metric_mask = 0
        for m in self.order:
            self.metric_mask |= L.M_BITS[m]
        self.thresholds = dict(thresholds)
        self.threshold_mask = 0
        for name, bit in L.T_BITS.items():
            if self.thresholds.get(name) is not None:
                self.threshold_mask |= bit
        h = dict(DEFAULT_HARM if harm_coeffs is None else harm_coeffs)
        self.harm = L.FoHarmCoeffs(*[float(h[k]) for k in ("rs_const", "rs_speed", "rs_side", "rs_rear", "ia_const",
                                                           "ia_speed", "ped_const", "ped_speed")])
        self.origin = np.zeros(2)
        self.agents: Optional[AgentSet] = None
        self._table = None
        self._corr = False            # the table is a correlated one (fo_agents_pack_corr / fo_metric_bundle_corr)
        self._raw_dev = None
        self.n_agents = 0
        self.t_stride = 0
        self._pack_pending = False    # agents adopted without their table (_adopt_agents): packed by the next launch
        self._batch = None
        self._staging = None          # page-locked staging of assess_batch's host bundles
        self._staging_done = None

    # ------------------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_agents(self, agents: AgentSet, origin=None):
        """Upload + pack the phantom predictions (once per planning cycle).  ``origin`` (x, y) is
        subtracted in float64 from agent and ego positions before the cast to float32."""
        self._adopt_agents(agents, origin)
        self._pack_agents()

    def _adopt_agents(self, agents: AgentSet, origin=None):
        """The host side of ``set_agents``: the engine takes ``agents`` and ``origin`` as its own, and the next launch
        that needs their table packs it (for results computed elsewhere, e.g. by ``batch.prefetch_interfaces``)."""
        self.agents = agents
        self.origin = np.zeros(2) if origin is None else np.asarray(origin, dtype=np.float64)
        A, Tp = agents.n_agents, agents.t_stride
        self.n_agents, self.t_stride = A, Tp
        self._table = None
        self._corr = False
        self._pack_pending = False
        if A == 0 or Tp == 0:
            self.n_agents = 0
            return
        if Tp > L.FO_MAX_STATES:
            raise ValueError(f"predictions longer than {L.FO_MAX_STATES} states are not supported")
        self._pack_pending = True

    def _pack_agents(self):
        """Upload + pack the adopted agents' table, if it is not packed yet."""
        if not self._pack_pending:
            return
        self._pack_pending = False
        agents, A, Tp = self.agents, self.n_agents, self.t_stride
        corr = agents.cov_xy is not None
        rows = [agents.x - self.origin[0], agents.y - self.origin[1], agents.yaw, agents.v, agents.var_x, agents.var_y]
        fl = np.stack(rows + ([agents.cov_xy] if corr else [])).astype(np.float32)
        pa = np.stack([agents.length, agents.width, agents.buf_length, agents.buf_width]).astype(np.float32)
        ia = np.stack([agents.n_states, agents.kind]).astype(np.int32)
        with torch.cuda.device(self.device):
            d_fl = torch.from_numpy(fl).to(self.device, non_blocking=False)
            d_pa = torch.from_numpy(pa).to(self.device)
            d_ia = torch.from_numpy(ia).to(self.device)
            raw = L.FoAgentsRaw()
            raw.n_agents, raw.t_stride = A, Tp
            raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y = [d_fl[i].data_ptr() for i in range(6)]
            raw.n_states, raw.kind = d_ia[0].data_ptr(), d_ia[1].data_ptr()
            raw.length, raw.width, raw.buf_length, raw.buf_width = [d_pa[i].data_ptr() for i in range(4)]
            if corr:
                nbytes = L.lib.fo_agent_table_bytes_corr(A, Tp)
                self._table = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
                L.check(L.lib.fo_agents_pack_corr(C.byref(raw), C.c_void_p(d_fl[6].data_ptr()), C.byref(self.vehicle),
                                                  C.c_void_p(self._table.data_ptr()), nbytes, self._stream()),
                        "fo_agents_pack_corr")
            else:
                nbytes = L.lib.fo_agent_table_bytes(A, Tp)
                self._table = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
                L.check(L.lib.fo_agents_pack(C.byref(raw), C.byref(self.vehicle), C.c_void_p(self._table.data_ptr()),
                                             nbytes, self._stream()), "fo_agents_pack")
            self._corr = corr
            self._raw_dev = (d_fl, d_pa, d_ia)  # keep alive until the stream work is done

    # ------------------------------------------------------------------------------------------
    def to_device_bundle(self, ego, origin=None) -> torch.Tensor:
        """[N, T, 5] -> contiguous float32 CUDA tensor (origin-shifted when given as host float64).  ``origin``: (x, y)
        for every trajectory, or an [N, 2] array of one origin per trajectory; default the agents' origin."""
        origin = self.origin if origin is None else np.asarray(origin, dtype=np.float64)
        per_row = origin.ndim == 2
        if isinstance(ego, torch.Tensor) and ego.is_cuda:
            t = ego
            if np.any(origin != 0.0):
                # device tensors are in the caller's frame: shift them like the agents (float64 offset vector)
                off = np.zeros((origin.shape[0], 1, 5) if per_row else (5,))
                off[..., 0], off[..., 1] = (origin[:, None, 0], origin[:, None, 1]) if per_row else (origin[0], origin[1])
                t = (t.to(torch.float64) - torch.from_numpy(off).to(t.device)).to(torch.float32)
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(torch.float32).contiguous()
            return t
        arr = np.array(ego, dtype=np.float64, copy=True)
        if arr.ndim == 2:
            arr = arr[None]
        arr[..., 0] -= origin[:, None, 0] if per_row else origin[0]
        arr[..., 1] -= origin[:, None, 1] if per_row else origin[1]
        host = torch.from_numpy(arr.astype(np.float32))
        if host.numel() >= (1 << 18):          # page-locking only pays for bundles of a megabyte and more
            return host.pin_memory().to(self.device, non_blocking=True)
        return host.to(self.device)

    def _args(self, t, out):
        N, T = int(t.shape[0]), int(t.shape[1])
        a = L.FoMetricArgs()
        a.ego, a.n_traj, a.n_states = t.data_ptr(), N, T
        a.agent_table = self._table.data_ptr() if self._table is not None else None
        a.n_agents, a.t_stride = self.n_agents, max(self.t_stride, 1)
        a.vehicle, a.harm, a.dt = self.vehicle, self.harm, self.dt
        a.metric_mask, a.threshold_mask = self.metric_mask, self.threshold_mask
        for name in L.T_BITS:
            v = self.thresholds.get(name)
            setattr(a, "thr_" + name, float(v) if v is not None else 0.0)
        a.valid, a.summary, a.flags = out.valid.data_ptr(), out.summary.data_ptr(), out.flags.data_ptr()
        deltas = out.peer_delta                        # parallel.PeerResultGatherer: fused result exchange
        if deltas:
            a.n_peers = len(deltas)
            for i, d in enumerate(deltas):
                a.peer_delta[i] = int(d)
        return a

    def work_stats(self, ego, correlated: bool = False) -> dict:
        """How much of the algorithmic work survives the exact bounds (``fo_metric_stats``): counts of visited
        (trajectory, agent, step) evaluations, exact box distances, LR4S logits, CP evaluations, BE pairs and pair
        tests (probes), BE tree nodes walked and re-timed ego-path chunks computed for one pass over ``ego``.  Used by
        bench.py's flop model; synchronises.

        ``correlated``: a set with correlated prediction covariances is counted by ``fo_metric_stats_corr``, which costs
        one pass of the correlated summary path (many times the diagonal one, DESIGN.md §5.10).  The counters do not
        depend on the covariances, so they equal those of the same set with ``cov_xy = None`` (in multi-warp team shapes
        "obb", "lr4s", "be" and "be_probes" vary from run to run on either path, DESIGN.md §5.13).  Without the flag
        such a set raises ``ValueError``; with it a diagonal set is counted exactly as without it."""
        corr = self.agents is not None and self.agents.cov_xy is not None and self.n_agents > 0
        if corr and not correlated:
            raise ValueError("work_stats() takes diagonal prediction covariances only unless correlated=True")
        t = self.to_device_bundle(ego)
        N = int(t.shape[0])
        dev = self.device
        self._pack_agents()
        with torch.cuda.device(dev):
            out = BundleResult(torch.empty(N, dtype=torch.uint8, device=dev),
                               torch.empty((N, L.FO_SUMMARY_K), dtype=torch.float32, device=dev),
                               torch.empty(N, dtype=torch.int32, device=dev))
            a = self._args(t, out)
            cnt = torch.zeros(10, dtype=torch.int64, device=dev)   # FO_STATS_K
            fn = "fo_metric_stats_corr" if self._corr else "fo_metric_stats"
            L.check(getattr(L.lib, fn)(C.byref(a), C.c_void_p(cnt.data_ptr()), self._stream()), fn)
            c = cnt.cpu().tolist()
        return {"visited": c[0], "obb": c[1], "lr4s": c[2], "cp": c[3], "be": c[4], "be_probes": c[5],
                "windows": c[6], "windows_kept": c[7], "be_nodes": c[8], "be_path_chunks": c[9]}

    def assess(self, ego, want_pair: bool = False, want_step: bool = False, out: Optional[BundleResult] = None
               ) -> BundleResult:
        """One pass of the dense core over a trajectory bundle (asynchronous on the current stream)."""
        t = self.to_device_bundle(ego)
        if t.ndim != 3 or t.shape[2] != 5:
            raise ValueError("trajectory bundle must have shape [N, T, 5] (x, y, theta, v, a)")
        N, T = int(t.shape[0]), int(t.shape[1])
        if T > L.FO_MAX_STATES:
            raise ValueError(f"trajectories longer than {L.FO_MAX_STATES} states are not supported")
        A = self.n_agents
        dev = self.device
        self._pack_agents()
        with torch.cuda.device(dev):
            if out is None:
                out = BundleResult(torch.empty(N, dtype=torch.uint8, device=dev),
                                   torch.empty((N, L.FO_SUMMARY_K), dtype=torch.float32, device=dev),
                                   torch.empty(N, dtype=torch.int32, device=dev))
                if want_pair:
                    out.pair = torch.empty((N, A, L.FO_PAIR_K), dtype=torch.float32, device=dev)
                if want_step:
                    out.step = torch.empty((N, A, max(T - 1, 0), L.FO_STEP_K), dtype=torch.float32, device=dev)
            a = self._args(t, out)
            a.pair = out.pair.data_ptr() if (out.pair is not None and A > 0) else None
            a.step = out.step.data_ptr() if (out.step is not None and A > 0 and T > 1) else None
            # a correlated table with peer stores (parallel.PeerResultGatherer) takes the call that honours them
            fn = ("fo_metric_bundle_corr_peers" if out.peer_delta else "fo_metric_bundle_corr") if self._corr \
                else "fo_metric_bundle"
            L.check(getattr(L.lib, fn)(C.byref(a), self._stream()), fn)
        out._keepalive = t
        return out

    def capture(self, ego_dev: torch.Tensor, out: Optional[BundleResult] = None):
        """CUDA-graph form of ``assess`` for the per-planning-step latency path: the launch on a device-resident
        bundle (fixed address and shape; refill it in place before every replay) is captured once, ``replay()``
        re-issues it without any per-call host work.  Returns ``(graph, out)``."""
        if not (isinstance(ego_dev, torch.Tensor) and ego_dev.is_cuda and ego_dev.dtype == torch.float32
                and ego_dev.is_contiguous()):
            raise ValueError("capture() needs a contiguous float32 CUDA tensor [N, T, 5]")
        N = int(ego_dev.shape[0])
        dev = self.device
        with torch.cuda.device(dev):
            if out is None:
                out = BundleResult(torch.empty(N, dtype=torch.uint8, device=dev),
                                   torch.empty((N, L.FO_SUMMARY_K), dtype=torch.float32, device=dev),
                                   torch.empty(N, dtype=torch.int32, device=dev))
            self.assess(ego_dev, out=out)                  # warm-up outside the capture (first-use attribute calls)
            torch.cuda.current_stream(dev).synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.assess(ego_dev, out=out)
        return g, out

    # ---- batches of independent problems ------------------------------------------------------------------------
    def set_agent_batch(self, agent_sets: Sequence[AgentSet], origins=None, vehicles=None, correlated: bool = False):
        """Upload + pack the phantom predictions of P independent problems (``fo_agents_pack_batch``): one float64
        origin shift per problem, one host-to-device copy of all of them, one pack call.  ``origins``: [P, 2] or None
        (no shift).  ``vehicles``: P ego vehicle descriptions (each a dict or an object with attributes, as the
        constructor takes them), or None for the engine's own vehicle in every problem; ``assess_batch`` assesses
        problem p with vehicles[p].  Problem p's table equals what ``set_agents(agent_sets[p], origins[p])`` packs in an
        engine built with vehicles[p].

        ``correlated``: sets with correlated prediction covariances (``AgentSet.cov_xy`` set) are accepted and packed
        as ``set_agents`` packs them (``fo_agents_pack_batch_corr``); their collision probabilities cost many times the
        diagonal ones.  Without it such a set raises ``ValueError``.  A batch without one makes the diagonal calls."""
        P = len(agent_sets)
        if not correlated and any(a.cov_xy is not None for a in agent_sets):
            raise ValueError("batches take diagonal prediction covariances only unless correlated=True; assess a "
                             "correlated set with set_agents() + assess()")
        veh = None
        if vehicles is not None:
            if len(vehicles) != P:
                raise ValueError(f"{len(vehicles)} vehicles for {P} problems")
            veh = (L.FoVehicle * max(P, 1))(*[vehicle_struct(v) for v in vehicles])
        org = np.zeros((P, 2)) if origins is None else np.asarray(origins, dtype=np.float64).reshape(P, 2)
        n_agents = np.array([a.n_agents if a.t_stride > 0 else 0 for a in agent_sets], dtype=np.int32)
        t_stride = np.array([a.t_stride if n else 0 for a, n in zip(agent_sets, n_agents)], dtype=np.int32)
        if np.any(t_stride > L.FO_MAX_STATES):
            raise ValueError(f"predictions longer than {L.FO_MAX_STATES} states are not supported")
        # the correlated problems (with agents, as set_agents packs them); None = the diagonal calls
        corr = np.array([a.cov_xy is not None and n > 0 for a, n in zip(agent_sets, n_agents)], dtype=np.uint8)
        corr = corr if corr.any() else None
        if corr is not None and veh is None:
            veh = (L.FoVehicle * P)(*[self.vehicle] * P)
        offsets = np.zeros(P, dtype=np.int64)
        if corr is None:
            arena_bytes = L.lib.fo_agent_batch_layout(P, n_agents.ctypes.data, t_stride.ctypes.data, offsets.ctypes.data)
        else:
            arena_bytes = L.lib.fo_agent_batch_layout_corr(P, n_agents.ctypes.data, t_stride.ctypes.data,
                                                           corr.ctypes.data, offsets.ctypes.data)
        problems = (L.FoBatchProblem * max(P, 1))()
        for p in range(P):
            problems[p].n_agents, problems[p].t_stride, problems[p].table_offset = int(n_agents[p]), int(t_stride[p]), int(offsets[p])
        A, S = int(n_agents.sum()), int(t_stride.max(initial=0))
        dev = self.device
        self._batch = {"problems": problems, "P": P, "origins": org, "agents": list(agent_sets), "arena": None,
                       "arena_bytes": arena_bytes, "n_agents": n_agents, "vehicles": veh, "corr": corr}
        if A == 0:
            return
        # one host buffer: 6 float rows [A, S] (x, y shifted per problem; a seventh, cov_xy, with correlated problems),
        # 4 float columns [A], 2 int32 columns [A]
        R = 6 if corr is None else 7
        buf = np.zeros(R * A * S + 6 * A, dtype=np.float32)
        fl = buf[:R * A * S].reshape(R, A, S)
        pa = buf[R * A * S:R * A * S + 4 * A].reshape(4, A)
        ia = buf[R * A * S + 4 * A:].view(np.int32).reshape(2, A)
        a0 = 0
        for p, ag in enumerate(agent_sets):
            n, tp = int(n_agents[p]), int(t_stride[p])
            if n == 0:
                continue
            rows = slice(a0, a0 + n)
            fl[0, rows, :tp] = ag.x - org[p, 0]
            fl[1, rows, :tp] = ag.y - org[p, 1]
            fl[2, rows, :tp], fl[3, rows, :tp], fl[4, rows, :tp], fl[5, rows, :tp] = ag.yaw, ag.v, ag.var_x, ag.var_y
            if corr is not None and corr[p]:
                fl[6, rows, :tp] = ag.cov_xy
            pa[:, rows] = (ag.length, ag.width, ag.buf_length, ag.buf_width)
            ia[:, rows] = (ag.n_states, ag.kind)
            a0 += n
        with torch.cuda.device(dev):
            host = torch.from_numpy(buf)
            d_buf = host.pin_memory().to(dev, non_blocking=True) if buf.nbytes >= (1 << 20) else host.to(dev)
            ptr, f4 = d_buf.data_ptr(), 4
            raw = L.FoAgentsRaw()
            raw.n_agents, raw.t_stride = A, S
            raw.x, raw.y, raw.yaw, raw.v, raw.var_x, raw.var_y = [ptr + f4 * i * A * S for i in range(6)]
            base = ptr + f4 * R * A * S
            raw.length, raw.width, raw.buf_length, raw.buf_width = [base + f4 * i * A for i in range(4)]
            raw.n_states, raw.kind = base + f4 * 4 * A, base + f4 * 5 * A
            arena = torch.empty(max(arena_bytes, 16), dtype=torch.uint8, device=dev)
            if corr is not None:
                L.check(L.lib.fo_agents_pack_batch_corr(C.byref(raw), C.c_void_p(ptr + f4 * 6 * A * S), P, problems,
                                                        corr.ctypes.data, veh, C.c_void_p(arena.data_ptr()), arena_bytes,
                                                        self._stream()), "fo_agents_pack_batch_corr")
            elif veh is None:
                L.check(L.lib.fo_agents_pack_batch(C.byref(raw), P, problems, C.byref(self.vehicle),
                                                   C.c_void_p(arena.data_ptr()), arena_bytes, self._stream()),
                        "fo_agents_pack_batch")
            else:
                L.check(L.lib.fo_agents_pack_batch_vehicles(C.byref(raw), P, problems, veh, C.c_void_p(arena.data_ptr()),
                                                            arena_bytes, self._stream()), "fo_agents_pack_batch_vehicles")
        self._batch["arena"] = arena
        self._batch["raw_dev"] = d_buf           # keep alive until the stream work is done

    def _stage_host_batch(self, parts, origins, offsets, T) -> torch.Tensor:
        """Host bundles of a batch -> one float32 device tensor: each problem shifted by its origin in float64 and
        written straight into a page-locked staging buffer kept by the engine (grown on demand; before it is refilled
        the copy out of it is waited for), then one asynchronous upload."""
        n = int(offsets[-1]) * T * 5
        if self._staging is None or self._staging.numel() < n:
            self._staging = torch.empty(n + n // 4, dtype=torch.float32).pin_memory()
            self._staging_done = None
        if self._staging_done is not None:
            self._staging_done.synchronize()
        view = self._staging.numpy()[:n].reshape(-1, T, 5)
        for p, e in enumerate(parts):
            lo, hi = int(offsets[p]), int(offsets[p + 1])
            if hi == lo:
                continue
            e = e.reshape(-1, T, 5)
            view[lo:hi] = e                              # same values as to_device_bundle: float64 shift, then float32
            view[lo:hi, :, 0] = e[..., 0] - origins[p, 0]
            view[lo:hi, :, 1] = e[..., 1] - origins[p, 1]
        t = self._staging[:n].view(-1, T, 5).to(self.device, non_blocking=True)
        self._staging_done = torch.cuda.Event()
        self._staging_done.record(torch.cuda.current_stream(self.device))
        return t

    def assess_batch(self, egos: Sequence, want_pair: bool = False, want_step: bool = False,
                     out: Optional[BatchResult] = None) -> BatchResult:
        """One pass over every problem of the batch set by ``set_agent_batch`` in one metric call.  ``egos[p]``: problem
        p's [N_p, T, 5] bundle (host array or CUDA tensor, in the caller's frame: it is shifted by the problem's origin).
        Without detail outputs this is ``fo_metric_batch``; with ``want_pair`` / ``want_step`` it is
        ``fo_metric_batch_detail`` (their ``_corr`` forms when the batch has a correlated problem), and ``split()`` gives problem p what ``set_agents`` + ``assess(want_pair,
        want_step)`` gives it alone (in an engine built with its vehicle, when ``set_agent_batch`` had ``vehicles``).
        ``out``: preallocated outputs of the batch's sizes (valid / summary / flags, and
        the flat pair / step where wanted).  Asynchronous on the current stream."""
        b = self._batch
        if b is None:
            raise RuntimeError("assess_batch() needs set_agent_batch() first")
        P = b["P"]
        if len(egos) != P:
            raise ValueError(f"{len(egos)} bundles for {P} problems")
        on_dev = [isinstance(e, torch.Tensor) and e.is_cuda for e in egos]
        if any(on_dev) and not all(on_dev):
            raise ValueError("bundles of one batch are either all CUDA tensors or all host arrays")
        if all(on_dev) and P:
            parts = [e if e.ndim == 3 else e[None] for e in egos]
        else:
            parts = [np.asarray(e.cpu() if isinstance(e, torch.Tensor) else e, dtype=np.float64) for e in egos]
            parts = [e if e.ndim == 3 else e[None] for e in parts]
        shapes = {tuple(e.shape[1:]) for e in parts if e.shape[0] > 0}
        if len(shapes) > 1 or any(s[1] != 5 for s in shapes):
            raise ValueError(f"every bundle must be [N_p, T, 5] with one T for the batch, got {sorted(shapes)}")
        T = shapes.pop()[0] if shapes else max([int(e.shape[1]) for e in parts], default=1)
        if T > L.FO_MAX_STATES:
            raise ValueError(f"trajectories longer than {L.FO_MAX_STATES} states are not supported")
        counts = np.array([int(e.shape[0]) for e in parts], dtype=np.int64)
        offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        N = int(offsets[-1])
        dev = self.device
        row_origin = np.repeat(b["origins"], counts, axis=0)
        n_pairs = int(np.dot(counts, b["n_agents"].astype(np.int64))) if P else 0
        with torch.cuda.device(dev):
            if N and all(on_dev):
                t = self.to_device_bundle(torch.cat([e.reshape(-1, T, 5) for e in parts]), origin=row_origin)
            elif N:
                t = self._stage_host_batch(parts, b["origins"], offsets, T)
            else:
                t = torch.empty((0, T, 5), dtype=torch.float32, device=dev)
            if out is None:
                out = BatchResult(torch.empty(N, dtype=torch.uint8, device=dev),
                                  torch.empty((N, L.FO_SUMMARY_K), dtype=torch.float32, device=dev),
                                  torch.empty(N, dtype=torch.int32, device=dev), offsets)
                if want_pair:
                    out.pair = torch.empty(n_pairs * L.FO_PAIR_K, dtype=torch.float32, device=dev)
                if want_step:
                    out.step = torch.empty(n_pairs * max(T - 1, 0) * L.FO_STEP_K, dtype=torch.float32, device=dev)
            out.offsets, out.n_agents, out.n_states = offsets, b["n_agents"], T
            if not want_pair:
                out.pair = None
            if not want_step:
                out.step = None
            problems = b["problems"]
            for p in range(P):
                problems[p].traj_begin, problems[p].n_traj = int(offsets[p]), int(counts[p])
            a = L.FoMetricBatchArgs()
            a.common = self._args(t, BundleResult(out.valid, out.summary, out.flags))
            a.common.agent_table = b["arena"].data_ptr() if b["arena"] is not None else None
            a.common.n_agents, a.common.t_stride = 0, 1
            a.n_problems, a.problems, a.arena_bytes = P, problems, b["arena_bytes"]
            # a problem without agents or a horizon of one state has no detail to write: as in assess, the summary
            # path runs when no detail buffer is left
            a.common.pair = out.pair.data_ptr() if (out.pair is not None and out.pair.numel()) else None
            a.common.step = out.step.data_ptr() if (out.step is not None and out.step.numel()) else None
            detail, veh, corr = bool(a.common.pair or a.common.step), b["vehicles"], b["corr"]
            if corr is not None:
                fn = "fo_metric_batch_detail_corr" if detail else "fo_metric_batch_corr"
                L.check(getattr(L.lib, fn)(C.byref(a), corr.ctypes.data, veh, self._stream()), fn)
            elif veh is None:
                fn = "fo_metric_batch_detail" if detail else "fo_metric_batch"
                L.check(getattr(L.lib, fn)(C.byref(a), self._stream()), fn)
            else:
                fn = "fo_metric_batch_detail_vehicles" if detail else "fo_metric_batch_vehicles"
                L.check(getattr(L.lib, fn)(C.byref(a), veh, self._stream()), fn)
        out._keepalive = (t, b["arena"])
        return out
