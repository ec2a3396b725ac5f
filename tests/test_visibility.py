"""Stage 1 / stage 2: oracle self-consistency on CPU, CUDA parity on the GPU."""
import numpy as np
import pytest

from frenetix_occlusion_b200 import synthetic as S
from oracle import visibility_oracle as VO


def _frame(seed, n_obst, with_ring=False, transparent_every=0, half_extent=40.0):
    rng = np.random.default_rng(seed)
    rect = S.obstacle_frames(1, n_obst, seed=seed, half_extent=half_extent)[0].astype(np.float64)
    # keep the ego outside every rectangle
    keep = np.hypot(rect[:, 0], rect[:, 1]) > 3.5
    flags = np.where(keep, VO.RECT_EXISTS, 0).astype(np.uint8)
    if transparent_every:
        flags[::transparent_every] |= VO.RECT_TRANSPARENT
    ego = np.array([0.0, 0.0, rng.uniform(-np.pi, np.pi)])
    boundary = None
    if with_ring:
        ang = np.linspace(0, 2 * np.pi, 101)
        rad = 35.0 + 6.0 * np.sin(3 * ang)
        pts = np.stack((rad * np.cos(ang), rad * np.sin(ang)), -1)
        boundary = np.concatenate((pts[:-1], pts[1:]), 1)
    return ego, rect, flags, boundary


@pytest.mark.parametrize("seed,n_obst,ring,fov", [(1, 12, False, 360.0), (2, 30, True, 360.0), (3, 20, False, 120.0),
                                                  (4, 8, True, 200.0)])
def test_raycast_oracle_agrees_with_reference_shadow_construction(seed, n_obst, ring, fov):
    """Polar first-hit map == point-wise evaluation of the reference's shadow-quad construction,
    outside a band of one angular step around shadow borders."""
    ego, rect, flags, boundary = _frame(seed, n_obst, ring)
    R, n_rays = 50.0, 4096
    rng_, hit, _ = VO.raycast(ego, rect, flags, boundary, R, fov, n_rays)
    ang = VO.ray_angles(ego[2], fov, n_rays)
    prng = np.random.default_rng(seed + 100)
    pr = np.sqrt(prng.uniform(0.04, 1.0, 6000)) * R * 0.995
    k = prng.integers(1, n_rays - 2, 6000)
    frac = prng.uniform(0.2, 0.8, 6000)
    pa = ang[k] + frac * (ang[1] - ang[0])
    P = ego[:2] + np.stack((pr * np.cos(pa), pr * np.sin(pa)), -1)
    ref = VO.reference_point_visible(P, ego, rect, flags, boundary, R, fov)
    lo = np.minimum(rng_[k], rng_[k + 1])
    hi = np.maximum(rng_[k], rng_[k + 1])
    tol = 0.02
    must_vis = pr < lo - tol
    must_occ = pr > hi + tol
    # the reference removes the obstacle polygon itself as well; points inside an obstacle are beyond the hit
    assert ref[must_vis].all(), f"{(~ref[must_vis]).sum()} points the ray map calls visible are shadowed in the reference"
    assert (~ref[must_occ]).all(), f"{ref[must_occ].sum()} points the ray map calls occluded are visible in the reference"
    assert must_vis.sum() > 500 and must_occ.sum() > 500


def test_rollout_oracle_kat():
    r = VO.rollout_cv([12.0], [-3.0], [1.4], [np.pi / 2], 0.1, 3.0)
    assert r["x"].shape == (1, 31)
    assert np.allclose(r["x"][0], 12.0) and np.isclose(r["y"][0, 30], -3.0 + 3.0 * 1.4)
    assert np.isclose(r["var"][0, 30], 0.1 * 1.05 ** 30)
    r = VO.rollout_cv([0.0], [0.0], [1.4], [0.3], 0.1, 3.0)
    assert np.isclose(r["x"][0, 10], round(1.4 * np.cos(0.3), 3))      # SURVEY.md 8c: round(1.4 cos phi, 3)


def _f32_frame(seed, n_obst, ring, transp):
    ego, rect, flags, boundary = _frame(seed, n_obst, ring, transp, half_extent=50.0)
    f32 = lambda a: None if a is None else a.astype(np.float32).astype(np.float64)
    return f32(ego), f32(rect), flags, f32(boundary)


@pytest.mark.parametrize("seed,n_obst,ring,fov,n_rays,transp", [(11, 64, False, 360.0, 4096, 0), (13, 40, True, 360.0, 1000, 5),
                                                                  (14, 25, True, 90.0, 333, 3), (15, 300, False, 200.0, 2048, 7),
                                                                  (17, 2000, False, 360.0, 256, 0)])
def test_certificate_accepts_float32_restatement(seed, n_obst, ring, fov, n_rays, transp):
    """The float32 restatement of the kernel's arithmetic (no culls) passes the float64 certificate on every ray."""
    ego, rect, flags, boundary = _f32_frame(seed, n_obst, ring, transp)
    r, h, v = VO.raycast_f32(ego, rect, flags, boundary, 50.0, fov, n_rays)
    cert = VO.certify_raycast(r, h, v, ego, rect, flags, boundary, 50.0, fov, n_rays)
    assert cert["n_fail"] == 0, VO.certificate_failures(cert)


def test_certificate_rejects_wrong_answers():
    """Each single wrong answer fails the certificate on the ray or obstacle it touches."""
    ego, rect, flags, boundary = _f32_frame(13, 40, True, 5)
    R, fov, n = 50.0, 360.0, 1000
    r, h, v = VO.raycast_f32(ego, rect, flags, boundary, R, fov, n)
    cert = lambda r_, h_, v_: VO.certify_raycast(r_, h_, v_, ego, rect, flags, boundary, R, fov, n)
    assert cert(r, h, v)["n_fail"] == 0
    hits = np.flatnonzero(h >= 0)
    owners = np.unique(h[hits])
    assert len(hits) > 50 and len(owners) > 2
    for k in hits[::len(hits) // 7]:
        r2, h2 = r.astype(np.float64), h.copy()
        r2[k], h2[k] = np.float32(R), VO.HIT_NONE                     # the hit dropped
        c = cert(r2, h2, None)
        assert not c["ray_ok"][k] and c["n_fail"] == 1, (k, VO.certificate_failures(c))
        r2 = r.astype(np.float64)
        r2[k] += 0.01                                                  # the range 1 cm long
        c = cert(r2, h, None)
        assert not c["ray_ok"][k] and c["n_fail"] == 1, (k, VO.certificate_failures(c))
        h2 = h.copy()
        h2[k] = owners[owners != h[k]][0]                              # the owner swapped
        c = cert(r, h2, None)
        assert not c["ray_ok"][k], (k, VO.certificate_failures(c))
    exists = (flags & VO.RECT_EXISTS) != 0
    transp = exists & ((flags & VO.RECT_TRANSPARENT) != 0)
    hidden = np.flatnonzero(exists & ~transp & (v == 0))
    seen_tr = np.flatnonzero(transp & (v == 1))
    assert len(hidden) and len(seen_tr)
    for o in hidden:                                                   # a hidden obstacle marked visible
        v2 = v.copy()
        v2[o] = 1
        c = cert(r, h, v2)
        assert not c["vis_ok"][o] and c["n_fail"] == 1, (o, VO.certificate_failures(c))
    for o in seen_tr:                                                  # a seen transparent obstacle's flag cleared
        v2 = v.copy()
        v2[o] = 0
        c = cert(r, h, v2)
        assert not c["vis_ok"][o] and c["n_fail"] == 1, (o, VO.certificate_failures(c))
    o = owners[0]                                                      # a hit obstacle's flag cleared
    v2 = v.copy()
    v2[o] = 0
    assert not cert(r, h, v2)["vis_ok"][o]


def test_oracle_ego_on_edge_rule():
    """An ego standing on a rectangle side is blocked at range 0 by exactly the rays that point to the box's side of
    it (at a corner: of either side); a zero-width box blocks both sides; a border segment through the ego blocks
    nothing, whichever way it is listed."""
    R, n = 50.0, 16
    ego = np.array([0.0, 0.0, 0.1])
    ang = VO.ray_angles(0.1, 360.0, n)
    d = np.stack((np.cos(ang), np.sin(ang)), -1)
    one = np.ones(1, np.uint8)
    for cx, cy, hl, hw in ((2.0, 1.0, 2.0, 1.0), (0.0, 1.0, 2.0, 1.0), (-2.0, -1.0, 2.0, 1.0), (0.0, 0.0, 2.0, 0.0)):
        rect = np.array([[cx, cy, 0.0, hl, hw]])
        rng, hit, vis = VO.raycast(ego, rect, one, None, R, 360.0, n)
        # inward normals of the sides through the ego (axis-aligned box, yaw 0)
        inward = [np.array(v) for on, v in ((cx - hl == 0, (1, 0)), (cx + hl == 0, (-1, 0)), (cy - hw == 0, (0, 1)),
                                            (cy + hw == 0, (0, -1))) if on]
        assert inward
        toward = np.any([d @ v > 0 for v in inward], 0)
        blocked = rng == 0
        if hw == 0:
            assert blocked.all()
        else:
            assert np.array_equal(blocked, toward), (cx, cy, blocked.astype(int), toward.astype(int))
        assert (hit[blocked] == 0).all() and vis[0] == 1
        r32, h32, _ = VO.raycast_f32(ego, rect, one, None, R, 360.0, n)
        assert np.array_equal(r32 == 0, blocked) and np.array_equal(h32, hit)
    seg = np.array([[-5.0, 0.0, 5.0, 0.0]])
    for b in (seg, seg[:, [2, 3, 0, 1]]):
        rng, hit, _ = VO.raycast(ego, np.zeros((0, 5)), np.zeros(0, np.uint8), b, R, 360.0, n)
        assert (rng == R).all() and (hit == VO.HIT_NONE).all()
        r32, h32, _ = VO.raycast_f32(ego, np.zeros((0, 5)), np.zeros(0, np.uint8), b, R, 360.0, n)
        assert (r32 == np.float32(R)).all() and (h32 == VO.HIT_NONE).all()


# ------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("seed,n_obst,ring,fov,n_rays,transp", [(11, 64, False, 360.0, 4096, 0), (12, 512, False, 360.0, 4096, 0),
                                                                  (13, 40, True, 360.0, 1000, 5), (14, 25, True, 90.0, 333, 3),
                                                                  (15, 300, False, 200.0, 2048, 7), (16, 0, True, 360.0, 512, 0),
                                                                  (17, 2000, False, 360.0, 256, 0)])
def test_cuda_raycast_matches_oracle(seed, n_obst, ring, fov, n_rays, transp, cuda_device):
    """Every ray and every visible flag of three frames per case passes the float64 certificate."""
    from vis_cert import cast, certify
    frames = []
    for f in range(3):
        frames.append(_frame(seed * 10 + f, n_obst, ring, transp, half_extent=50.0))
    ego = np.stack([fr[0] for fr in frames])
    ego[:, :2] += np.array([[3.0, -2.0], [0.0, 0.0], [-7.5, 4.25]])      # non-trivial ego positions
    rect = np.stack([fr[1] for fr in frames]).reshape(3, n_obst, 5)
    rect[..., :2] += ego[:, None, :2]
    flags = np.stack([fr[2] for fr in frames]).reshape(3, n_obst)
    boundary = frames[0][3]
    R = 50.0
    # inputs rounded to float32 so both sides see identical numbers
    ego, rect = ego.astype(np.float32).astype(np.float64), rect.astype(np.float32).astype(np.float64)
    if boundary is not None:
        boundary = boundary.astype(np.float32).astype(np.float64)
    out = cast(ego, rect, flags, boundary, R, fov, n_rays)
    for f in range(3):
        certify(out, f, ego[f], rect[f], flags[f], boundary, R, fov, n_rays)


@pytest.mark.gpu
def test_cuda_rollout_cv_matches_oracle(cuda_device):
    from frenetix_occlusion_b200.prediction import rollout_cv
    import torch
    rng = np.random.default_rng(3)
    A = 37
    x0, y0 = rng.uniform(-50, 50, A), rng.uniform(-50, 50, A)
    v, phi = rng.uniform(0.5, 12, A), rng.uniform(-np.pi, np.pi, A)
    for horizon in (3.0, 5.0):
        r = rollout_cv(x0, y0, v, phi, 0.1, horizon)
        torch.cuda.synchronize()
        o = VO.rollout_cv(x0, y0, v, phi, 0.1, horizon)
        for key in ("x", "y", "yaw", "v", "var"):
            g = r[key].cpu().numpy()
            assert g.shape == o[key].shape
            assert np.array_equal(g, o[key].astype(np.float32)), key     # correctly rounded image of the float64 values


def _arc_path(radius, n=200, length=120.0):
    s = np.linspace(0, length, n)
    return np.stack((radius * np.sin(s / radius), radius * (1 - np.cos(s / radius))), -1)


def test_path_rollout_oracle_invariants():
    """Invariants that hold regardless of the un-vendored frenetix arithmetic: on a straight path with zero
    lateral offset the constant-speed, d1 = 0 sample has zero speed variance and reproduces CV exactly."""
    path = np.stack((np.linspace(-10, 100, 56), np.zeros(56)), -1)
    r = VO.rollout_path(path, 5.0, 0.0, 10.0, 0.1, 3.0)
    assert r["sample"] == 4                                   # speed factor 1.0, d1 = 0
    assert np.allclose(r["x"], 5.0 + 10.0 * np.arange(31) * 0.1, atol=1e-9) and np.allclose(r["y"], 0.0, atol=1e-12)
    assert np.allclose(r["v"], 10.0) and np.allclose(r["yaw"], 0.0)
    # lateral offset 0.4 m: nearest target offset is +0.5, speed stays ~constant, ends at d = 0.5
    r = VO.rollout_path(path, 5.0, 0.4, 10.0, 0.1, 3.0)
    assert r["sample"] == 5 and abs(r["y"][-1] - 0.5) < 1e-9 and abs(r["d0"] - 0.4) < 1e-12
    # circular arc: radius preserved for d = 0
    arc = _arc_path(40.0)
    r = VO.rollout_path(arc, arc[10, 0], arc[10, 1], 8.0, 0.1, 3.0)
    rad = np.hypot(r["x"], r["y"] - 40.0)
    assert np.all(np.abs(rad - 40.0) < 0.01)
    # low-velocity mode (v0 < 0.5 m/s, frenetix_handler.py:91-95): the lateral offset is a function of the covered arc
    # length -- an agent that stands still (v0 = 0: every sample has end speed 0) does not move sideways either
    r = VO.rollout_path(path, 5.0, 0.4, 0.0, 0.1, 3.0)
    assert np.allclose(r["x"], 5.0) and np.allclose(r["y"], 0.4) and np.allclose(r["v"], 0.0)
    r = VO.rollout_path(path, 5.0, 0.4, 0.3, 0.1, 3.0)
    assert abs(r["y"][0] - 0.4) < 1e-12 and np.all(np.diff(r["x"]) > 0) and np.all(np.abs(r["y"] - 0.4) <= 0.9 + 1e-9)


@pytest.mark.gpu
def test_cuda_path_rollout_matches_oracle(cuda_device):
    from frenetix_occlusion_b200.prediction import rollout_path
    import torch
    rng = np.random.default_rng(8)
    paths = [np.stack((np.linspace(-10, 100, 56), np.zeros(56)), -1), _arc_path(40.0), _arc_path(-25.0, 300, 150.0),
             np.stack((np.linspace(0, 60, 31), 3.0 * np.sin(np.linspace(0, 60, 31) / 9.0)), -1)]
    paths.append(paths[0])                                  # low-velocity mode: v0 < 0.5 m/s
    x0 = [5.0, 9.0, 3.0, 12.0, 7.0]
    y0 = [0.4, 1.5, -0.3, 2.2, 0.3]
    v0 = [10.0, 8.0, 5.0, 10.0, 0.3]
    for horizon in (3.0, 5.0):
        g = rollout_path(paths, x0, y0, v0, 0.1, horizon)
        torch.cuda.synchronize()
        for j, p in enumerate(paths):
            o = VO.rollout_path(p, x0[j], y0[j], v0[j], 0.1, horizon)
            assert int(g["sample"][j]) == o["sample"], (j, int(g["sample"][j]), o["sample"])
            for key in ("x", "y", "yaw", "v", "var"):
                np.testing.assert_allclose(g[key][j].cpu().numpy(), o[key], rtol=2e-6, atol=2e-5, err_msg=f"{key} job {j}")


@pytest.mark.gpu
def test_full_size_visibility_sweep_properties(cuda_device):
    """BASELINE.json configs[4] at FULL size (10,000 frames x 4096 rays x 512 rectangles): frame-sharding and
    obstacle-order invariance of the ray cast, and two frames against the float64 oracle."""
    import torch
    from frenetix_occlusion_b200.visibility import raycast_frames
    from vis_cert import assert_same_or_tied, certify
    F, R, O = S.C_VIS["n_frames"], S.C_VIS["n_rays"], S.C_VIS["n_obstacles"]
    rect = torch.from_numpy(S.obstacle_frames(F, O)).cuda()
    flags = torch.ones((F, O), dtype=torch.uint8, device="cuda")
    ego = torch.zeros((F, 3), dtype=torch.float32, device="cuda")
    ego[:, 2] = torch.linspace(-3.0, 3.0, F, device="cuda")
    whole = raycast_frames(ego, rect, flags, None, 50.0, 360.0, R)
    torch.cuda.synchronize()
    h = F // 2
    a = raycast_frames(ego[:h], rect[:h], flags[:h], None, 50.0, 360.0, R)
    b = raycast_frames(ego[h:], rect[h:], flags[h:], None, 50.0, 360.0, R)
    torch.cuda.synchronize()
    # Ranges are bit-identical across sharding and obstacle order.  Should that ever fail, it would have to be at an
    # exact corner tie (``t.x < bq * D`` is not exactly a minimum of quotients, so the staging order of a frame's edges
    # can matter there): the differing rays must then each pass the certificate and differ by at most 2 ulp.
    assert torch.equal(torch.cat((a.range, b.range)).view(torch.int32), whole.range.view(torch.int32))
    # where two obstacles' edges meet a ray at the same float32 range (crossing rectangles), either may be reported as
    # the owner -- the staging order of a frame's edges is not fixed: every differing answer must pass the certificate
    host = lambda t: t.cpu().numpy()
    rect_h, ego_h = host(rect).astype(np.float64), host(ego).astype(np.float64)
    frame = lambda f: (ego_h[f], rect_h[f], np.ones(O, np.uint8), None)
    whole_h = (host(whole.range), host(whole.hit), host(whole.visible))
    assert_same_or_tied(whole_h, tuple(host(torch.cat((u, v))) for u, v in ((a.range, b.range), (a.hit, b.hit),
                                                                            (a.visible, b.visible))),
                        frame, 50.0, 360.0, R, what="sharded")
    # the instrumented twin (fo_visibility_stats) writes the same outputs, and its counters nest as the culls do
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    c = raycast_frames(ego, rect, flags, None, 50.0, 360.0, R, stats=cnt)
    torch.cuda.synchronize()
    assert torch.equal(c.range.view(torch.int32), whole.range.view(torch.int32))
    tested, skipped, staged, listed = cnt.cpu().tolist()
    assert 0 < staged <= F * 4 * O and 0 < listed <= staged * (R // 256)
    assert tested + 32 * skipped <= listed * 256 and 0 < tested < F * R * 4 * O
    perm = torch.randperm(O, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    p = raycast_frames(ego, rect[:, perm].contiguous(), flags[:, perm].contiguous(), None, 50.0, 360.0, R)
    torch.cuda.synchronize()
    assert torch.equal(p.range.view(torch.int32), whole.range.view(torch.int32))          # first-hit distance: a min
    assert torch.equal(p.visible, whole.visible[:, perm])
    inv = torch.argsort(perm)
    mapped = torch.where(p.hit >= 0, perm[p.hit.clamp(min=0).long()].to(torch.int32), p.hit)
    assert_same_or_tied(whole_h, (host(p.range), host(mapped), host(p.visible[:, inv])), frame, 50.0, 360.0, R,
                        what="permuted")
    for f in (0, F - 1):
        certify(whole_h, f, ego_h[f], rect_h[f], np.ones(O, np.uint8), None, 50.0, 360.0, R)
