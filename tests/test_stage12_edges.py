"""Stage 1 / stage 2 kernels at their edges: the path-following rollout (``fo_rollout_path``) against ``VO.rollout_path``
and on properties that need no oracle, and the spawn rasters (``fo_spawn_region`` / ``fo_spawn_rect``) against
scipy.ndimage and a numpy restatement on masks of known topology.  The point classifier's edge cases extend
``test_scenarios.test_cuda_point_classification_matches_oracle``.

Reference-only checks (no marker) run on the CPU; the kernel comparisons are marked ``gpu``."""
import ctypes as C

import numpy as np
import pytest

from oracle import visibility_oracle as VO

RTOL, ATOL = 2e-6, 2e-5            # float32 outputs of a float64 evaluation (as test_visibility's path rollout test)
KEYS = ("x", "y", "yaw", "v", "var")


# ================================================================================================ path rollout
def _polyline(xy, heading=0.0, origin=(0.0, 0.0)):
    c, s = np.cos(heading), np.sin(heading)
    xy = np.asarray(xy, dtype=np.float64)
    return np.stack((xy[:, 0] * c - xy[:, 1] * s, xy[:, 0] * s + xy[:, 1] * c), -1) + np.asarray(origin)


def _wiggle(n, step, amp, period, heading=0.0, x_start=0.0):
    x = x_start + step * np.arange(n)
    return _polyline(np.stack((x, amp * np.sin(2 * np.pi * x / period)), -1), heading)


def _hairpin():
    """North-bound approach, a left semicircle of radius 8 m (segment headings pi/2 -> pi -> -pi/2), south-bound exit."""
    th = np.linspace(0.0, np.pi, 41)
    arc = np.stack((-8.0 + 8.0 * np.cos(th), 8.0 * np.sin(th)), -1)
    approach = np.stack((np.zeros(10), np.linspace(-20.0, -2.0, 10)), -1)
    exit_ = np.stack((np.full(10, -16.0), np.linspace(-2.0, -20.0, 10)), -1)
    return np.concatenate((approach, arc, exit_))


def _at(path, u, lateral):
    """Point at fractional vertex index u of ``path``, ``lateral`` metres to the left of that segment."""
    j = min(int(np.floor(u)), len(path) - 2)
    e = path[j + 1] - path[j]
    t = e / np.hypot(*e)
    p = path[j] + (u - j) * e
    return p[0] - lateral * t[1], p[1] + lateral * t[0]


def _oracle_jobs():
    """(path, x0, y0, v0, label) of every oracle-comparison case."""
    jobs = []
    long = _wiggle(1024, 0.5, 2.0, 40.0, heading=0.3, x_start=-255.0)       # 32 scan chunks
    for u in (0.1, 31.5, 511.5, 1019.5):                                    # near vertex 0, chunk boundaries, the end
        jobs.append((long, *_at(long, u, 0.3), 10.0, f"1024 vertices, start at vertex {u}"))
    straight = _polyline(np.stack((2.0 * np.arange(30), np.zeros(30)), -1), heading=1.1)
    t = np.array([np.cos(1.1), np.sin(1.1)])
    n = np.array([-t[1], t[0]])
    p = straight[0] - 4.0 * t + 0.2 * n
    jobs.append((straight, p[0], p[1], 8.0, "start before the first vertex"))
    p = straight[-1] + 3.0 * t - 0.3 * n
    jobs.append((straight, p[0], p[1], 8.0, "start beyond the last vertex"))
    jobs.append((straight, *_at(straight, 25.5, 0.4), 15.0, "horizon carries the agent past the end"))
    hp = _hairpin()
    jobs.append((hp, 0.3, -12.0, 8.0, "hairpin through heading pi"))
    jobs.append((_wiggle(200, 0.5, 0.3, 6.0, heading=np.pi), -10.0, 0.2, 10.0, "segment headings wiggle around pi"))
    u_path = np.array([[0.0, 0.0], [10.0, 0.0], [20.0, 0.0], [20.0, 4.0], [10.0, 4.0], [0.0, 4.0]])
    jobs.append((u_path, 7.0, 2.0, 5.0, "start equidistant from two segments"))
    curve = _wiggle(80, 1.0, 1.5, 50.0, heading=-0.7)
    for v0 in (0.0, 0.4999, 0.5, 0.5001):                                   # the 0.5 m/s low-velocity switch
        jobs.append((curve, *_at(curve, 10.3, -0.3), v0, f"v0 = {v0}"))
    return jobs


def _repeat_variants(path):
    """``path`` with repeated and sub-millimetre vertices inserted: each variant must give the same rollout.  A vertex
    within 1 mm of its predecessor is dropped, so an inserted near-copy goes right after the vertex it copies."""
    rng = np.random.default_rng(5)
    n = len(path)

    def near(k):                      # 0.2 .. 0.9 mm away from vertex k, in a random direction
        a, r = rng.uniform(-np.pi, np.pi), rng.uniform(2e-4, 9e-4)
        return path[k] + r * np.array([np.cos(a), np.sin(a)])

    ins = lambda k, *rows: np.concatenate((path[:k + 1], np.array(rows), path[k + 1:]))   # noqa: E731  (after vertex k)
    return {"first vertex repeated": np.concatenate((path[:1], path)),
            "vertex 20 repeated": ins(20, path[20]),
            "vertex 7 three times": ins(7, path[7], path[7]),
            "last vertex repeated": ins(n - 1, path[-1]),
            "last vertex repeated twice": ins(n - 1, path[-1], path[-1]),
            "sub-mm vertex after vertex 3": ins(3, near(3)),
            "sub-mm vertices after vertex 12 and 13": np.concatenate((path[:13], [near(12)], path[13:14], [near(13)], path[14:])),
            "sub-mm vertex after the last": ins(n - 1, near(n - 1)),
            "repeats everywhere": np.repeat(path, 2, axis=0)}


def _repeat_bases():
    """(path, x0, y0, v0): the straight north-bound path of 2 m steps (with a vertex repeated, its selected sample used to
    change), a curve, and starts from which the horizon carries the agent past the path end (a repeated last vertex
    used to freeze it at the end point)."""
    north = np.stack((np.zeros(30), 2.0 * np.arange(30)), -1)
    curve = _wiggle(60, 1.0, 2.0, 30.0, heading=0.4)
    return [(north, -0.4, 5.0, 10.0), (north, 0.3, 40.0, 10.0), (curve, *_at(curve, 3.2, 0.4), 9.0),
            (curve, *_at(curve, 40.5, -0.2), 6.0), (curve, *_at(curve, 20.5, 0.1), 0.3)]


def test_rollout_oracle_ignores_repeated_vertices():
    """VO.rollout_path: repeated and sub-millimetre vertices anywhere, at both ends, leave the rollout bit-identical."""
    for path, x0, y0, v0 in _repeat_bases():
        base = VO.rollout_path(path, x0, y0, v0, 0.1, 5.0)
        assert base["sample"] >= 0
        for name, p in _repeat_variants(path).items():
            r = VO.rollout_path(p, x0, y0, v0, 0.1, 5.0)
            assert r["sample"] == base["sample"], (name, r["sample"], base["sample"])
            for key in KEYS:
                assert np.array_equal(r[key], base[key]), (name, key)


def test_rollout_oracle_degenerate_paths():
    """Fewer than 2 vertices left after dropping repeats: sample -1 and zero rows."""
    for p in (np.zeros((0, 2)), np.array([[3.0, 4.0]]), np.array([[3.0, 4.0]] * 5), np.array([[3.0, 4.0], [3.0, 4.0005]])):
        r = VO.rollout_path(p, 3.0, 4.0, 5.0, 0.1, 3.0)
        assert r["sample"] == -1 and all(np.array_equal(r[k], np.zeros(int(3.0 / 0.1) + 1)) for k in KEYS)


def _rotate(xy, a):
    c, s = np.cos(a), np.sin(a)
    xy = np.asarray(xy, dtype=np.float64)
    return np.stack((xy[..., 0] * c - xy[..., 1] * s, xy[..., 0] * s + xy[..., 1] * c), -1)


def _rotation_jobs():
    """Paths near the origin (float32 rounding of the rotated vertices stays well under the tolerance)."""
    curve = _wiggle(60, 1.0, 2.0, 30.0, heading=0.0, x_start=-20.0)
    hp = _hairpin()
    return [(curve, *_at(curve, 5.5, 0.3), 9.0), (hp, 0.3, -12.0, 8.0), (curve, *_at(curve, 50.5, -0.2), 6.0)]


def _check_rotation(run):
    """``run(paths, x0, y0, v0)`` -> list of rollouts; rotating the inputs by a rotates x, y and shifts yaw by a."""
    jobs = _rotation_jobs()
    base = run([j[0] for j in jobs], [j[1] for j in jobs], [j[2] for j in jobs], [j[3] for j in jobs])
    for a in (0.7, np.pi / 2, 2.9, -2.2):
        st = _rotate(np.array([[j[1], j[2]] for j in jobs]), a)
        rot = run([_rotate(j[0], a) for j in jobs], st[:, 0], st[:, 1], [j[3] for j in jobs])
        for k, (b, r) in enumerate(zip(base, rot)):
            assert r["sample"] == b["sample"], (a, k)
            want = _rotate(np.stack((b["x"], b["y"]), -1), a)
            np.testing.assert_allclose(r["x"], want[:, 0], rtol=RTOL, atol=ATOL, err_msg=f"x, a={a}, job {k}")
            np.testing.assert_allclose(r["y"], want[:, 1], rtol=RTOL, atol=ATOL, err_msg=f"y, a={a}, job {k}")
            dyaw = (np.asarray(r["yaw"], np.float64) - b["yaw"] - a + np.pi) % (2 * np.pi) - np.pi
            assert np.all(np.abs(dyaw) <= ATOL + RTOL * np.abs(b["yaw"])), (a, k, np.abs(dyaw).max())
            for key in ("v", "var"):
                np.testing.assert_allclose(r[key], b[key], rtol=RTOL, atol=ATOL, err_msg=f"{key}, a={a}, job {k}")


def test_rollout_oracle_rotation_invariance():
    _check_rotation(lambda P, X, Y, V: [VO.rollout_path(p, x, y, v, 0.1, 5.0) for p, x, y, v in zip(P, X, Y, V)])


# ------------------------------------------------------------------------------------------------ GPU
def _gpu_rollout(paths, x0, y0, v0, dt, horizon, origin=(0.0, 0.0)):
    import torch
    from frenetix_occlusion_b200.prediction import rollout_path
    g = rollout_path(paths, x0, y0, v0, dt, horizon, origin=origin)
    torch.cuda.synchronize()
    out = {k: g[k].cpu().numpy() for k in KEYS}
    out["sample"] = g["sample"].cpu().numpy()
    return out


def _row(g, j):
    return {**{k: g[k][j] for k in KEYS}, "sample": int(g["sample"][j])}


def _assert_matches(row, o, what):
    assert row["sample"] == o["sample"], (what, row["sample"], o["sample"])
    for key in KEYS:
        np.testing.assert_allclose(row[key], o[key], rtol=RTOL, atol=ATOL, err_msg=f"{key}: {what}")


@pytest.mark.gpu
@pytest.mark.parametrize("n_states,dt", [(1, 0.125), (31, 0.125), (32, 0.125), (33, 0.125), (51, 0.125), (51, 0.1)])
def test_cuda_path_rollout_edges_match_oracle(n_states, dt, cuda_device):
    """Every edge case in one call: long paths, extrapolation at both ends, running past the end, headings across
    +-pi, an equidistant start and the low-velocity switch; horizons around the 32-lane step loop."""
    horizon = (n_states - 1) * dt
    assert int(horizon / dt) + 1 == n_states
    jobs = _oracle_jobs()
    g = _gpu_rollout([j[0] for j in jobs], [j[1] for j in jobs], [j[2] for j in jobs], [j[3] for j in jobs], dt, horizon)
    assert g["x"].shape == (len(jobs), n_states)
    for k, (path, x0, y0, v0, what) in enumerate(jobs):
        _assert_matches(_row(g, k), VO.rollout_path(path, x0, y0, v0, dt, horizon), what)


@pytest.mark.gpu
def test_cuda_path_rollout_per_job_origins(cuda_device):
    """Paths and starts at ~1e5 m, one origin per job (subtracted in float64 before the float32 cast)."""
    jobs = _oracle_jobs()
    rng = np.random.default_rng(11)
    org = rng.uniform(0.8e5, 1.2e5, (len(jobs), 2))
    g = _gpu_rollout([j[0] + org[k] for k, j in enumerate(jobs)], [j[1] + org[k, 0] for k, j in enumerate(jobs)],
                     [j[2] + org[k, 1] for k, j in enumerate(jobs)], [j[3] for j in jobs], 0.1, 5.0, origin=org)
    for k, (path, x0, y0, v0, what) in enumerate(jobs):
        _assert_matches(_row(g, k), VO.rollout_path(path, x0, y0, v0, 0.1, 5.0), what)


@pytest.mark.gpu
def test_cuda_path_rollout_ignores_repeated_vertices(cuda_device):
    """The kernel drops vertices within 1 mm of their predecessor: every variant is bit-identical to its base path."""
    paths, x0, y0, v0, names = [], [], [], [], []
    for b, (path, x, y, v) in enumerate(_repeat_bases()):
        for name, p in [("base", path)] + list(_repeat_variants(path).items()):
            paths.append(p); x0.append(x); y0.append(y); v0.append(v); names.append((b, name))
    g = _gpu_rollout(paths, x0, y0, v0, 0.1, 5.0)
    base = {}
    for k, (b, name) in enumerate(names):
        if name == "base":
            base[b] = k
            assert g["sample"][k] >= 0
            _assert_matches(_row(g, k), VO.rollout_path(paths[k], x0[k], y0[k], v0[k], 0.1, 5.0), f"base {b}")
            continue
        ref = base[b]
        assert g["sample"][k] == g["sample"][ref], (b, name)
        for key in KEYS:
            assert np.array_equal(g[key][k], g[key][ref]), (b, name, key)


@pytest.mark.gpu
def test_cuda_path_rollout_rotation_invariance(cuda_device):
    def run(P, X, Y, V):
        g = _gpu_rollout(P, X, Y, V, 0.1, 5.0)
        return [_row(g, k) for k in range(len(P))]
    _check_rotation(run)


@pytest.mark.gpu
def test_cuda_path_rollout_batch_equals_single_jobs(cuda_device):
    """512 jobs in one launch are bit-identical to the same jobs launched one at a time."""
    rng = np.random.default_rng(17)
    paths, x0, y0, v0 = [], [], [], []
    for k in range(512):
        n = int(rng.choice([2, 3, 31, 32, 33, 200, 1024]))
        p = _wiggle(n, rng.uniform(0.3, 3.0), rng.uniform(0.0, 3.0), rng.uniform(10.0, 80.0), heading=rng.uniform(-np.pi, np.pi),
                    x_start=rng.uniform(-30.0, 0.0))
        paths.append(p)
        x, y = _at(p, rng.uniform(-1.0, n - 0.5), rng.uniform(-1.0, 1.0))
        x0.append(x); y0.append(y); v0.append(float(rng.choice([0.0, 0.3, 0.5, rng.uniform(1.0, 20.0)])))
    whole = _gpu_rollout(paths, x0, y0, v0, 0.1, 5.0)
    for k in range(512):
        one = _gpu_rollout(paths[k:k + 1], x0[k:k + 1], y0[k:k + 1], v0[k:k + 1], 0.1, 5.0)
        assert one["sample"][0] == whole["sample"][k], k
        for key in KEYS:
            assert np.array_equal(one[key][0], whole[key][k]), (k, key)


@pytest.mark.gpu
def test_cuda_path_rollout_padding_and_degenerate_paths(cuda_device):
    """Direct C-ABI call with t_stride = n_states + 7 into NaN-filled outputs: the padding columns are written with
    zeros; paths of 0 and 1 vertex (and of one vertex repeated) give sample -1 and all-zero rows."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    curve = _wiggle(40, 1.0, 1.5, 20.0, heading=0.2)
    paths = [curve, np.zeros((0, 2)), np.array([[1.0, 2.0]]), np.array([[1.0, 2.0]] * 4), curve[::-1].copy()]
    x0, y0, v0 = [3.0, 1.0, 1.0, 1.0, 30.0], [0.5, 2.0, 2.0, 2.0, 1.0], [7.0, 7.0, 7.0, 7.0, 4.0]
    J, T, dt, horizon = len(paths), 51, 0.1, 5.0
    S = T + 7
    dev = cuda_device
    off = np.concatenate(([0], np.cumsum([len(p) for p in paths]))).astype(np.int32)
    d_xy = torch.from_numpy(np.concatenate(paths).astype(np.float32)).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_st = torch.from_numpy(np.array([x0, y0, v0], dtype=np.float64)).to(dev)
    out = torch.full((6, J, S), float("nan"), dtype=torch.float32, device=dev)
    smp = torch.full((J,), 99, dtype=torch.int32, device=dev)
    a = L.FoRolloutPathArgs()
    a.n_jobs, a.n_states, a.t_stride, a.dt, a.t1, a.var0, a.var_factor = J, T, S, dt, 3.0, 0.1, 1.05
    a.path_xy, a.path_off = d_xy.data_ptr(), d_off.data_ptr()
    a.x0, a.y0, a.v0 = [d_st[i].data_ptr() for i in range(3)]
    a.x, a.y, a.yaw, a.vel, a.var_x, a.var_y = [out[i].data_ptr() for i in range(6)]
    a.sample = smp.data_ptr()
    L.check(L.lib.fo_rollout_path(C.byref(a), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "fo_rollout_path")
    torch.cuda.synchronize()
    o, s = out.cpu().numpy(), smp.cpu().numpy()
    assert not np.isnan(o).any()
    assert np.array_equal(o[:, :, T:], np.zeros((6, J, 7), np.float32))
    ref = _gpu_rollout([paths[0], paths[4]], [x0[0], x0[4]], [y0[0], y0[4]], [v0[0], v0[4]], dt, horizon)
    for k, r in ((0, 0), (4, 1)):
        assert s[k] == ref["sample"][r] >= 0
        for i, key in enumerate(KEYS):
            assert np.array_equal(o[i, k, :T], ref[key][r]), (k, key)
        assert np.array_equal(o[5, k, :T], o[4, k, :T])                        # var_y == var_x
    for k in (1, 2, 3):
        assert s[k] == -1 and not o[:, k].any(), k


# ================================================================================================ spawn rasters
# Synthetic masks are encoded as ONE lanelet ring, so the region predicate reduces to lanelet membership: every set run
# of cells along the first raster axis (runs with the same extent in consecutive rows merged) becomes a rectangle whose
# edges lie on cell boundaries, and the rectangles are joined by bridges -- horizontal segments along cell-boundary rows
# and a vertical line left of the raster.  Horizontal edges never count in the even-odd test and the bridge line lies
# left of every cell centre, so the crossing parity at a cell centre is exactly the mask.  Cell = 0.125 m and raster
# corners at integer metres from the frame origin: every cell boundary and centre is exact in float32.
CELL = 0.125
ORG = np.array([1000.0, -500.0])          # frame origin (world); the ego sits on it, heading +x toward the rasters


def _runs(mask):
    """Rectangles (i0, i1, j0, j1) (half-open cell ranges) that tile the set cells of ``mask`` [nx, ny]."""
    rects, live = [], {}
    for j in range(mask.shape[1]):
        d = np.diff(np.concatenate(([0], mask[:, j].astype(np.int8), [0])))
        nxt = {}
        for a, b in zip(np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]):
            k = live.get((a, b))
            if k is None:
                k = len(rects)
                rects.append([a, b, j, j + 1])
            else:
                rects[k][3] = j + 1
            nxt[(a, b)] = k
        live = nxt
    return rects


def mask_ring(mask, x0, y0):
    """The ring (frame coordinates) whose even-odd interior at the cell centres of a raster with lower-left corner
    (x0, y0) is ``mask``."""
    xl = x0 - 1.0
    ring = [(xl - 1.0, y0), (xl, y0), (xl, y0 + CELL)]      # an empty mask: a triangle left of the raster
    if mask.any():
        ring = []
    for i0, i1, j0, j1 in _runs(mask):
        xa, xb, ya, yb = x0 + i0 * CELL, x0 + i1 * CELL, y0 + j0 * CELL, y0 + j1 * CELL
        ring += [(xl, ya), (xa, ya), (xb, ya), (xb, yb), (xa, yb), (xa, ya), (xl, ya)]
    return np.array(ring, dtype=np.float64).reshape(-1, 2)


def _spiral(nx, ny, w=2):
    """One rectangular spiral of arm width w and gap w (a single part with very long union chains)."""
    m = np.zeros((nx, ny), bool)
    a0, b0, a1, b1 = 0, 0, nx, ny
    while a1 - a0 >= 3 * w and b1 - b0 >= 3 * w:
        m[a0:a1, b0:b0 + w] = True
        m[a1 - w:a1, b0:b1] = True
        m[a0:a1, b1 - w:b1] = True
        m[a0:a0 + w, b0 + 2 * w:b1] = True
        if a1 - a0 >= 7 * w and b1 - b0 >= 7 * w:
            m[a0 + w:a0 + 2 * w, b0 + 2 * w:b0 + 3 * w] = True         # connector into the next turn
        a0, b0, a1, b1 = a0 + 2 * w, b0 + 2 * w, a1 - 2 * w, b1 - 2 * w
    return m


def _comb(nx, ny, axis):
    """Teeth one cell wide, one cell apart, joined only by a spine at the far end of ``axis``."""
    m = np.zeros((nx, ny), bool)
    if axis == 1:
        m[::2, :] = True
        m[:, -1] = True
    else:
        m[:, ::2] = True
        m[-1, :] = True
    return m


def _equal_parts(nx, ny, k):
    """k parts of 12 cells of different shapes (the tie goes to the part first in raster order)."""
    m = np.zeros((nx, ny), bool)
    if nx == 1 or ny == 1:                      # bars along the only axis
        flat = m.reshape(-1)
        for p in range(k):
            flat[100 + 200 * p:112 + 200 * p] = True
        return m
    shapes = [np.ones((3, 4), bool), np.ones((1, 12), bool), np.array([[1] * 9, [1, 0, 0, 0, 0, 0, 0, 0, 0],
                                                                     [1, 0, 0, 0, 0, 0, 0, 0, 0], [1] + [0] * 8], bool)]
    at = [(nx - 10, 5), (nx // 2, ny // 2), (3, ny - 12)]    # raster order: the L (i = 3) comes first
    for p in range(k):
        s = shapes[p]
        m[at[p][0]:at[p][0] + s.shape[0], at[p][1]:at[p][1] + s.shape[1]] |= s
    return m


def _border(nx, ny):
    """A frame along every raster border with a cross through the middle, and a separate small part inside."""
    m = np.zeros((nx, ny), bool)
    m[0, :] = m[-1, :] = m[:, 0] = m[:, -1] = True
    m[nx // 2, :] = m[:, ny // 2] = True
    m[3:6, 3:5] = True
    return m


def _shape(name, nx, ny):
    if name == "empty":
        return np.zeros((nx, ny), bool)
    if name == "full":
        return np.ones((nx, ny), bool)
    if name == "single":
        m = np.zeros((nx, ny), bool)
        m[nx // 3, ny // 3] = True
        return m
    if name == "checkerboard":
        return (np.add.outer(np.arange(nx), np.arange(ny)) % 2) == 0
    if name == "spiral":
        return _spiral(nx, ny)
    if name.startswith("comb"):
        return _comb(nx, ny, int(name[-1]))
    if name.startswith("equal"):
        return _equal_parts(nx, ny, int(name[-1]))
    if name == "border":
        return _border(nx, ny)
    raise KeyError(name)


REGION_CASES = [("empty", 240, 240), ("full", 240, 240), ("single", 240, 240), ("spiral", 240, 240), ("comb1", 240, 240),
                ("equal2", 240, 240), ("equal3", 240, 240), ("border", 240, 240), ("checkerboard", 48, 48),
                ("checkerboard", 1, 4096), ("full", 1, 4096), ("equal2", 1, 4096), ("checkerboard", 4096, 1),
                ("full", 4096, 1), ("equal3", 4096, 1), ("spiral", 257, 255), ("comb0", 257, 255), ("border", 257, 255),
                ("equal3", 257, 255), ("full", 1024, 1024), ("spiral", 1024, 1024), ("comb1", 1024, 1024)]


def _raster_frame(nx, ny):
    """Lower-left raster corner (frame coordinates, integer metres) and the cell centres (world, float64)."""
    x0, y0 = 8.0, -float(np.floor(ny * CELL / 2))
    cx = ORG[0] + x0 + 0.5 * nx * CELL
    cy = ORG[1] + y0 + 0.5 * ny * CELL
    gx = (np.arange(nx) + 0.5) * CELL - 0.5 * nx * CELL
    gy = (np.arange(ny) + 0.5) * CELL - 0.5 * ny * CELL
    X = np.broadcast_to((cx + gx)[:, None], (nx, ny))
    Y = np.broadcast_to((cy + gy)[None, :], (nx, ny))
    return x0, y0, cx, cy, X, Y


def _expected_region(mask, X, Y):
    """scipy.ndimage: 4-connected parts, the largest (first in raster order on ties), its one-cell dilation."""
    from scipy import ndimage
    lab, n = ndimage.label(mask)
    part = np.zeros_like(mask)
    if n:
        part = lab == 1 + int(np.argmax(ndimage.sum(mask, lab, np.arange(1, n + 1))))
    flat = lab.reshape(-1)
    root = np.full(flat.shape, -1, np.int64)
    nz = np.nonzero(flat)[0]
    if len(nz):
        ids, first = np.unique(flat[nz], return_index=True)
        lowest = np.zeros(n + 1, np.int64)
        lowest[ids] = nz[first]
        root[nz] = lowest[flat[nz]]
    return {"n": n, "part": part, "dilated": ndimage.binary_dilation(part), "root": root,
            "count": int(part.sum()), "sum_x": float(X[part].sum()), "sum_y": float(Y[part].sum())}


@pytest.mark.parametrize("name,nx,ny", [c for c in REGION_CASES if c[1] * c[2] <= 60000])
def test_mask_ring_encodes_the_mask(name, nx, ny):
    """Reference-only: the float64 even-odd test of the ring at every cell centre is the mask; shapes have the topology
    their names promise."""
    from scipy import ndimage
    mask = _shape(name, nx, ny)
    x0, y0, _, _, X, Y = _raster_frame(nx, ny)
    ring = mask_ring(mask, x0, y0)
    assert len(ring) < 20000
    inside = VO.points_in_polygon(np.stack((X - ORG[0], Y - ORG[1]), -1).reshape(-1, 2), ring) if len(ring) else \
        np.zeros(nx * ny, bool)
    assert np.array_equal(inside.reshape(nx, ny), mask)
    n = ndimage.label(mask)[1]
    want = {"empty": 0, "full": 1, "single": 1, "spiral": 1, "comb0": 1, "comb1": 1, "equal2": 2, "equal3": 3, "border": 2,
            "checkerboard": int(mask.sum())}[name]
    assert n == want, (name, n)


def _region_call(frame, nx, ny, cx, cy, disc, probe, ws):
    import torch
    from frenetix_occlusion_b200 import _lib as L
    a = L.FoSpawnRegionArgs()
    a.frame = frame._frame_args(-1, 0.0)
    a.raster = frame._raster_spec((cx, cy), 1.0, 0.0, 0.5 * nx * CELL, 0.5 * ny * CELL, CELL, nx, ny)
    a.pred = frame._predicate(1, L.PT_OCCLUDED, 0, disc[:2], disc[2])
    a.probe_x, a.probe_y = float(probe[0]), float(probe[1])
    a.label, a.size, a.best = ws["label"].data_ptr(), ws["size"].data_ptr(), ws["best"].data_ptr()
    a.mask_dilated, a.result = ws["dilated"].data_ptr(), ws["result"].data_ptr()
    L.check(L.lib.fo_spawn_region(C.byref(a), C.c_void_p(torch.cuda.current_stream(frame.device).cuda_stream)),
            "fo_spawn_region")
    torch.cuda.synchronize()
    r = L.FoRasterResult.from_buffer_copy(ws["result"].cpu().numpy().tobytes())
    return r, ws["label"].cpu().numpy(), ws["dilated"].cpu().numpy()


def _mask_frame(ring):
    from frenetix_occlusion_b200.visibility import FrameGeometry
    # sensor radius 1 mm: nothing is visible; occluded radius 1e4 m covers every raster
    return FrameGeometry(ORG, 0.0, np.zeros((0, 5)), np.zeros(0, np.uint8), None, [ring + ORG], 1e-3, 360.0,
                         occluded_factor=1e7)


@pytest.mark.gpu
@pytest.mark.parametrize("name,nx,ny", REGION_CASES + [("disc", 240, 240)])
def test_cuda_spawn_region_matches_scipy(name, nx, ny, cuda_device):
    """fo_spawn_region on masks of known topology against scipy.ndimage: part count, largest part (ties to the first
    in raster order), labels, dilation, area, centroid sums and probe answers."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    mask = _shape("spiral" if name == "disc" else name, nx, ny)
    x0, y0, cx, cy, X, Y = _raster_frame(nx, ny)
    frame = _mask_frame(mask_ring(mask, x0, y0))
    # the classification alone reproduces the mask (a classification fault cannot pass for a labelling fault)
    f, _, lan = frame.classify(np.stack((X, Y), -1).reshape(-1, 2))
    assert np.array_equal(((f & L.PT_OCCLUDED) != 0) & ((lan & np.uint64(1)) != 0), mask.reshape(-1))
    disc = (cx, cy, float(np.hypot(nx, ny) * CELL))                      # covers the raster
    if name == "disc":                                                  # cuts it
        disc = (cx - 9.0, cy + 4.0, 17.3)
        dd = np.hypot(X - disc[0], Y - disc[1])
        assert np.abs(dd - disc[2]).min() > 1e-6
        mask = mask & (dd <= disc[2])
    want = _expected_region(mask, X, Y)
    n = nx * ny
    ws = {"label": torch.empty(n, dtype=torch.int32, device=cuda_device), "size": torch.empty(n, dtype=torch.int32, device=cuda_device),
          "best": torch.zeros(1, dtype=torch.int64, device=cuda_device), "dilated": torch.empty(n, dtype=torch.uint8, device=cuda_device),
          "result": torch.zeros(32, dtype=torch.uint8, device=cuda_device)}
    # probes: exactly on lower-left cell corners (floor rule), cell centres of the chosen and of another part, the
    # upper-right corner of a part cell, and just outside every side
    lo_x, lo_y = ORG[0] + x0, ORG[1] + y0
    probes = [(lo_x - 1e-3, cy), (lo_x + nx * CELL, cy), (cx, lo_y - 1e-3), (cx, lo_y + ny * CELL), (lo_x, lo_y)]
    part_cells = np.argwhere(want["part"])
    if len(part_cells):
        i, j = part_cells[len(part_cells) // 2]
        probes += [(lo_x + i * CELL, lo_y + j * CELL), (X[i, j], Y[i, j]), (lo_x + (i + 1) * CELL, lo_y + (j + 1) * CELL)]
    other = np.argwhere(mask & ~want["part"])
    if len(other):
        i, j = other[len(other) // 3]
        probes += [(X[i, j], Y[i, j]), (lo_x + i * CELL, lo_y + j * CELL)]
    first = None
    for probe in probes:
        r, label, dil = _region_call(frame, nx, ny, cx, cy, disc, probe, ws)
        assert r.n_components == want["n"] and r.count == want["count"], (probe, r.n_components, r.count, want["n"], want["count"])
        fi, fj = np.floor((probe[0] - (cx - 0.5 * nx * CELL)) / CELL), np.floor((probe[1] - (cy - 0.5 * ny * CELL)) / CELL)
        inside = 0 <= fi < nx and 0 <= fj < ny and bool(want["part"][int(fi), int(fj)])
        assert r.contains == int(inside), (probe, fi, fj)
        if first is None:
            first = (label, dil)
            assert np.array_equal(label, want["root"]), int((label != want["root"]).sum())
            assert np.array_equal(dil.reshape(nx, ny) != 0, want["dilated"]) and set(np.unique(dil)) <= {0, 1}
            if want["count"]:
                assert abs(r.sum_x - want["sum_x"]) <= 1e-9 * abs(want["sum_x"])
                assert abs(r.sum_y - want["sum_y"]) <= 1e-9 * abs(want["sum_y"])
            else:
                assert r.sum_x == 0.0 and r.sum_y == 0.0
        else:                                       # the labelling does not depend on the schedule
            assert np.array_equal(label, first[0]) and np.array_equal(dil, first[1])


# ------------------------------------------------------------------------------------------------ candidate boxes
def _raster_points(cx, cy, cs, sn, hx, hy, cell, nx, ny):
    """fo_spawn.cu raster_point restated: same operation order, no fused multiply-adds.  [nx, ny] each."""
    gx = ((np.arange(nx) + 0.5) * cell - hx)[:, None]
    gy = ((np.arange(ny) + 0.5) * cell - hy)[None, :]
    return (cx + gx * cs) - gy * sn, (cy + gx * sn) + gy * cs


def _rect_expected(X, Y, region, rox, roy, rcell):
    rn = region.shape[0]
    fi, fj = np.floor((X - rox) / rcell), np.floor((Y - roy) / rcell)
    ok = (fi >= 0) & (fi < rn) & (fj >= 0) & (fj < rn)
    m = np.zeros(X.shape, bool)
    m[ok] = region[fi[ok].astype(int), fj[ok].astype(int)]
    p = np.pad(m, 1)
    core = p[1:-1, :-2] & p[1:-1, 2:] & p[:-2, 1:-1] & p[2:, 1:-1]
    return m, m & ~core


@pytest.mark.gpu
@pytest.mark.parametrize("deg", [0.0, 30.0, 90.0, -135.0])
def test_cuda_spawn_rect_matches_numpy(deg, cuda_device):
    """fo_spawn_rect on uploaded region masks: count and outline equal (as sets, bit for bit) to a numpy restatement,
    sums to 1e-9; centre_from records of count 2 (ignored) and 3 (centroid); an outline larger than its capacity."""
    import torch
    from scipy import ndimage
    from frenetix_occlusion_b200 import _lib as L
    rng = np.random.default_rng(int(deg) + 400)
    rn, rcell = 64, 0.25
    rox, roy = ORG[0] + 30.0, ORG[1] - 8.0
    region = ndimage.binary_opening(rng.random((rn, rn)) < 0.7)      # blobs with holes and ragged borders
    big = np.array([[-5.0, -200.0], [300.0, -200.0], [300.0, 200.0], [-5.0, 200.0]])   # road everywhere ahead
    frame = _mask_frame(big)
    dev = cuda_device
    d_region = torch.from_numpy(region.astype(np.uint8).reshape(-1)).to(dev)
    a_rad = np.radians(deg)
    cs, sn = np.cos(a_rad), np.sin(a_rad)
    length, width, cell = 5.5, 2.5, 0.025
    nx, ny = int(round(length / cell)), int(round(width / cell))
    C0 = (ORG[0] + 38.3, ORG[1] - 0.4)
    rec = L.FoRasterResult()
    rec.sum_x, rec.sum_y = 3 * (ORG[0] + 37.1), 3 * (ORG[1] + 0.9)
    for count, cap in ((None, 4096), (2, 4096), (3, 4096), (None, 7)):
        rec.count = count or 0
        d_rec = torch.from_numpy(np.frombuffer(bytes(rec), np.uint8).copy()).to(dev)
        mask_ws = torch.empty(nx * ny, dtype=torch.uint8, device=dev)
        outline = torch.full((max(cap, 1), 2), float("nan"), dtype=torch.float64, device=dev)
        res = torch.zeros(32, dtype=torch.uint8, device=dev)
        a = L.FoSpawnRectArgs()
        a.frame = frame._frame_args(-1, 0.0)
        a.raster = frame._raster_spec(C0, cs, sn, 0.5 * length, 0.5 * width, cell, nx, ny)
        a.pred = frame._predicate(1, L.PT_OCCLUDED, 0, C0, 50.0)
        a.centre_from = d_rec.data_ptr() if count else None
        a.region_mask, a.region_ox, a.region_oy, a.region_cell, a.region_n = d_region.data_ptr(), rox, roy, rcell, rn
        a.outline_cap, a.mask, a.outline, a.result = cap, mask_ws.data_ptr(), outline.data_ptr(), res.data_ptr()
        L.check(L.lib.fo_spawn_rect(C.byref(a), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "fo_spawn_rect")
        torch.cuda.synchronize()
        r = L.FoRasterResult.from_buffer_copy(res.cpu().numpy().tobytes())
        cx, cy = C0
        if count == 3:
            cx, cy = rec.sum_x / 3, rec.sum_y / 3
        X, Y = _raster_points(cx, cy, cs, sn, 0.5 * length, 0.5 * width, cell, nx, ny)
        m, edge = _rect_expected(X, Y, region, rox, roy, rcell)
        assert 100 < m.sum() < m.size, int(m.sum())                     # the box straddles the region's border
        assert np.array_equal(mask_ws.cpu().numpy().reshape(nx, ny) != 0, m)
        assert r.count == int(m.sum()) and r.n_outline == int(edge.sum()) and r.contains == 0 and r.n_components == 0
        assert abs(r.sum_x - X[m].sum()) <= 1e-9 * abs(X[m].sum()) and abs(r.sum_y - Y[m].sum()) <= 1e-9 * abs(Y[m].sum())
        want = {(x, y) for x, y in zip(X[edge], Y[edge])}
        got = outline.cpu().numpy()[:min(cap, r.n_outline)]
        got_set = {(x, y) for x, y in got}
        assert len(got_set) == len(got)                                 # no outline cell written twice
        if cap >= r.n_outline:
            assert got_set == want
        else:                                                           # capacity exceeded: a subset, full count
            assert len(got) == cap and got_set <= want
