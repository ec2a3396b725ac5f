"""Count model of the brake evaluation (BE) in the summary kernel, on the float64 oracle.

Every colliding pair of a trajectory bisects the required deceleration from the same bracket [lo0, 5] with the same
midpoint and stop rules (be.py:66-79), so all probes of a trajectory are nodes of one binary tree.  Only the maximum
over the pairs leaves the summary kernel.  This script runs two ways of getting that maximum and counts 32-step chunks:

  * per pair (be_bisect): one bisection per pair, in list order, each stopped once its bracket lies at or below the
    maximum so far (the floor) and no later probe can overrun the planned path;
  * tree walk (be_walk): the tree visited depth first, hit child first, with the re-timed ego path computed once per
    node and every pair that reaches the node tested against it; a pending node at or below the floor is dropped
    under the same overrun condition.

Both give the same maximum and the same range error (the reference raises when the re-timed path overruns the planned
one, be.py:117-124); tests/test_be_walk.py checks that.  No GPU needed.
usage: python scripts/be_tree_count.py [n_traj]"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import metric_oracle as MO  # noqa: E402

MARGIN = 0.99999       # the kernels' margin on the overrun test of a dropped bracket


class Trajectory:
    """The BE inputs of one trajectory: its re-timed paths (cached per deceleration) and the pair test."""

    def __init__(self, case, n, stacked):
        ego = np.asarray(case["ego"], dtype=np.float64)
        self.T = ego.shape[1]
        self.x, self.y, self.th, self.v, acc = (ego[n, :, k] for k in range(5))
        self.dist = np.insert(np.cumsum(np.sqrt(np.diff(self.x) ** 2 + np.diff(self.y) ** 2)), 0, 0)
        self.time = np.arange(self.T - 1) * case["dt"]
        self.dt = case["dt"]
        self.lo0 = np.round(abs(min(min(acc), 0)), 2)
        self.case, self.stacked = case, stacked
        self.cache = {}

    def length(self, cur):
        """dist_new[T-1] at deceleration cur"""
        v_new = np.insert(np.maximum(self.v[1] - cur * self.time, 0), 0, self.v[0:1])
        return np.cumsum(v_new * self.dt)[-2] if self.T > 1 else 0.0

    def path(self, cur):
        """re-timed ego box centre and heading, None when the re-timed path overruns the planned one"""
        if cur not in self.cache:
            v_new = np.insert(np.maximum(self.v[1] - cur * self.time, 0), 0, self.v[0:1])
            dn = np.insert(np.cumsum(v_new * self.dt), 0, 0)[:-1]
            if dn[-1] > self.dist[-1]:
                self.cache[cur] = None
            else:
                vp = self.case["vehicle"]
                xn, yn, tn = (np.interp(dn, self.dist, q) for q in (self.x, self.y, self.th))
                self.cache[cur] = (xn + vp["wb_rear_axle"] * np.cos(tn), yn + vp["wb_rear_axle"] * np.sin(tn), tn)
        return self.cache[cur]

    def test(self, a, cur):
        """(hit, 32-step chunks scanned with the per-chunk early exit); an agent without states counts as a hit"""
        A, Ta, Tm, pos, yaw, vel, var = self.stacked
        p = self.path(cur)
        nn = min(self.T, Ta[a])
        if nn == 0:
            return True, 0
        vp, ag = self.case["vehicle"], self.case["agents"][a]
        hit = MO.obb_intersects(p[0][:nn], p[1][:nn], p[2][:nn], vp["length"] / 2, vp["width"] / 2, pos[a, :nn, 0],
                                pos[a, :nn, 1], yaw[a, :nn], ag["length"] / 2, ag["width"] / 2)
        idx = np.flatnonzero(hit)
        return (True, idx[0] // 32 + 1) if len(idx) else (False, (nn + 31) // 32)

    def droppable(self, lo, hi, probes):
        """a bracket reached after `probes` probes: is the end of its all-miss branch safely inside the planned path?"""
        c = (lo + hi) / 2
        for _ in range(probes + 1, 10):
            if c - lo < 0.1:
                break
            c = (lo + c) / 2
        return self.length(c) < self.dist[-1] * MARGIN


def per_pair(tr, agents, floor=0.0):
    """be_bisect for each pair in turn with the running maximum as floor: (maximum, range error, counts)"""
    cnt = dict(probes=0, path_chunks=0)
    for a in agents:
        lo, hi = tr.lo0, 5.0
        for it in range(10):
            cur = (lo + hi) / 2
            cnt["probes"] += 1
            if tr.path(cur) is None:
                return floor, True, cnt
            hit, c = tr.test(a, cur)
            cnt["path_chunks"] += c
            if hit:
                lo = cur
            else:
                hi = cur
            if hi - lo < 0.1:
                break
            if hi <= floor and tr.droppable(lo, hi, it + 1):
                break
        floor = max(floor, cur)
    return floor, False, cnt


def tree_walk(tr, agents, floor=0.0):
    """be_walk: (maximum, range error, counts)"""
    cnt = dict(nodes=0, tests=0, path_chunks=0, test_chunks=0)
    stack = [(tr.lo0, 5.0, list(agents), 0)]
    while stack:
        lo, hi, grp, d = stack.pop()
        if d > 0 and hi <= floor and tr.droppable(lo, hi, d):
            continue
        cur = (lo + hi) / 2
        if tr.path(cur) is None:
            return floor, True, cnt
        cnt["nodes"] += 1
        hits, miss, chunks = [], [], 0
        for a in grp:
            hit, c = tr.test(a, cur)
            cnt["tests"] += 1
            cnt["test_chunks"] += c
            chunks = max(chunks, c)
            (hits if hit else miss).append(a)
        cnt["path_chunks"] += chunks
        for g, l2, h2 in ((miss, lo, cur), (hits, cur, hi)):     # the hit child is popped first
            if not g:
                continue
            if h2 - l2 < 0.1 or d + 1 == 10:
                floor = max(floor, cur)
            else:
                stack.append((l2, h2, g, d + 1))
    return floor, False, cnt


def be_pairs(case):
    """{trajectory: colliding pairs with ttc > 0} (be.py:49-50)"""
    ttc = MO.evaluate_bundle(dict(case, activated_metrics=["dce", "ttc"]), want_detail=False)["ttc"]
    pairs = np.argwhere(np.isfinite(ttc) & (ttc > 0))
    return {int(n): [int(a) for a in pairs[pairs[:, 0] == n][:, 1]] for n in np.unique(pairs[:, 0])}


def main():
    import bench
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 400
    case = bench.make_case(bench.workload("c-sweep"), n)
    stacked = MO._stack_agents(case)
    tot = dict(traj=0, pairs=0, pp_probes=0, pp_chunks=0, nodes=0, tests=0, path_chunks=0, test_chunks=0, err=0)
    for nidx, agents in be_pairs(case).items():
        tr = Trajectory(case, nidx, stacked)
        m0, e0, c0 = per_pair(tr, agents)
        m1, e1, c1 = tree_walk(tr, agents)
        assert e0 == e1 and (e0 or m0 == m1), (nidx, m0, m1, e0, e1)
        tot["traj"] += 1
        tot["pairs"] += len(agents)
        tot["err"] += e0
        tot["pp_probes"] += c0["probes"]
        tot["pp_chunks"] += c0["path_chunks"]
        for k in ("nodes", "tests", "path_chunks", "test_chunks"):
            tot[k] += c1[k]
    t, p = max(tot["traj"], 1), max(tot["pairs"], 1)
    print("%d trajectories of %d with BE, %.1f pairs each, %d range errors" % (tot["traj"], n, p / t, tot["err"]))
    print("per pair:  %.2f probes per pair, %.1f ego-path chunks per trajectory (one per pair-test chunk)"
          % (tot["pp_probes"] / p, tot["pp_chunks"] / t))
    print("tree walk: %.2f pair tests per pair, %.1f nodes and %.1f ego-path chunks per trajectory, %.1f pair-test chunks"
          % (tot["tests"] / p, tot["nodes"] / t, tot["path_chunks"] / t, tot["test_chunks"] / t))


if __name__ == "__main__":
    main()
