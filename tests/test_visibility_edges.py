"""The visibility ray cast (``fo_visibility_raycast``) at its edges, every answer held to the float64 certificate
``VO.certify_raycast``: launch shapes (fans per CTA, partial CTAs, more than 16 fans), 1024-edge tiles and the hit carried
between them, the angular cull and its 2 pi wrap, the distance rings and the sensor-disc cull, an ego on an edge,
transparent obstacles (listed and scanned), far origins, frame counts above the grid limit and invariances.  The
constant-velocity rollout of the same file (``fo_rollout_cv``) is held bit-exact to ``VO.rollout_cv`` on its edges.

Each case names the kernel path it exists for.  The C-ABI argument check runs on the CPU; everything else is ``gpu``."""
import ctypes as C

import numpy as np
import pytest

from oracle import visibility_oracle as VO
from vis_cert import assert_same_or_tied, cast, certify, f32

R = 50.0
EX, TR = VO.RECT_EXISTS, VO.RECT_EXISTS | VO.RECT_TRANSPARENT


def _clutter(rng, n, lo=4.0, hi=48.0, transparent_every=0):
    """n boxes at ego distances in [lo, hi] (ego at the origin), random yaw and size."""
    d, a = rng.uniform(lo, hi, n), rng.uniform(-np.pi, np.pi, n)
    rect = np.stack((d * np.cos(a), d * np.sin(a), rng.uniform(-np.pi, np.pi, n), rng.uniform(0.2, 2.5, n),
                     rng.uniform(0.2, 1.2, n)), -1)
    flags = np.full(n, EX, np.uint8)
    if transparent_every:
        flags[::transparent_every] = TR
    return rect, flags


def _ring(radius, n, amp=0.0, centre=(0.0, 0.0), a0=0.0, span=2 * np.pi):
    """n border segments along a (wavy) circle arc, as (x1, y1, x2, y2)."""
    ang = a0 + np.linspace(0.0, span, n + 1)
    rad = radius + amp * np.sin(3 * ang)
    pts = np.stack((centre[0] + rad * np.cos(ang), centre[1] + rad * np.sin(ang)), -1)
    return np.concatenate((pts[:-1], pts[1:]), 1)


def _check_frames(ego, rect, flags, boundary, fov, n_rays, what=""):
    """Cast frames ego [F,3] / rect [F,O,5] / flags [F,O] (float32-rounded here) and certify every frame."""
    ego, rect, boundary = f32(ego), f32(rect), f32(boundary)
    out = cast(ego, rect, flags, boundary, R, fov, n_rays)
    for f in range(len(ego)):
        certify(out, f, ego[f], rect[f], flags[f], boundary, R, fov, n_rays, what=what)
    return out


# ------------------------------------------------------------------------------------------------ launch shapes
def _pool():
    """Four frames sharing one border ring: clutter with transparent boxes, varied headings."""
    rng = np.random.default_rng(5)
    frames = [_clutter(rng, 60, transparent_every=6) for _ in range(4)]
    ego = np.array([[0.0, 0.0, -np.pi], [0.0, 0.0, 0.3], [0.0, 0.0, 2.0], [0.0, 0.0, 20 * np.pi]])
    return f32(ego), f32(np.stack([fr[0] for fr in frames])), np.stack([fr[1] for fr in frames]), f32(_ring(38.0, 100, 5.0))


@pytest.mark.gpu
@pytest.mark.parametrize("n_rays", [1, 31, 32, 33, 255, 256, 257, 4095, 4096, 4097, 8192])
def test_cuda_raycast_launch_shapes(n_rays, cuda_device):
    """Fans per CTA 1, 2, 4, 8 and 16 (chosen from the frame count against 4 x SMs), partial last CTAs, more than 16
    fans per frame: every frame equals its single-frame cast (fans per CTA 1), which passes the certificate; the
    instrumented twin (fo_visibility_stats) writes the same outputs."""
    import torch
    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    q = 4 * sms
    ego, rect, flags, bnd = _pool()
    single = []
    for p in range(4):
        out = cast(ego[p:p + 1], rect[p:p + 1], flags[p:p + 1], bnd, R, 360.0, n_rays)
        certify(out, 0, ego[p], rect[p], flags[p], bnd, R, 360.0, n_rays, what=f"single p={p}")
        single.append(out)
    frame = lambda f: (ego[f % 4], rect[f % 4], flags[f % 4], bnd)
    for F in (1, q // 8 - 1, q // 8, q // 4 - 1, q // 4, q // 2, q, q + 8):
        idx = np.arange(F) % 4
        stats = torch.zeros(4, dtype=torch.int64, device=cuda_device) if F in (q // 4, q + 8) else None
        out = cast(ego[idx], rect[idx], flags[idx], bnd, R, 360.0, n_rays, stats=stats)
        ref = tuple(np.stack([single[p][k][0] for p in idx]) for k in range(3))
        assert_same_or_tied(ref, out, frame, R, 360.0, n_rays, what=f"F={F}")
        if stats is not None:
            assert_same_or_tied(ref, cast(ego[idx], rect[idx], flags[idx], bnd, R, 360.0, n_rays), frame, R, 360.0,
                                n_rays, what=f"F={F} plain vs stats")
            assert stats[2].item() > 0


# ------------------------------------------------------------------------------------------------ tiles
@pytest.mark.gpu
@pytest.mark.parametrize("n_cand", [1023, 1024, 1025, 2048, 2049, 4097])
def test_cuda_raycast_tiles(n_cand, cuda_device):
    """Candidate counts around the 1024-edge tile, border only (rect NULL): the near occluder (a 3/4 arc at 8 m) in
    the last tiles and the far ring in the first, and the other way round -- the running hit is carried between tiles
    in the output slots.  With 256 boxes in front the border segments start in the second tile."""
    n_far = n_cand // 2
    far, near = _ring(40.0, n_far, 2.0), _ring(8.0, n_cand - n_far, 0.5, a0=0.3, span=1.5 * np.pi)
    ego = np.array([[0.0, 0.0, 0.7]])
    none = (np.zeros((1, 0, 5)), np.zeros((1, 0), np.uint8))
    for bnd in (np.concatenate((far, near)), np.concatenate((near, far))):
        out = _check_frames(ego, *none, bnd, 360.0, 2048, what=f"n_cand={n_cand}")
        assert (out[1] == VO.HIT_BOUNDARY).all()
    rect, flags = _clutter(np.random.default_rng(n_cand), 256, lo=10.0, hi=30.0)
    _check_frames(ego, rect[None], flags[None], np.concatenate((near, far)), 360.0, 2048, what="boxes + border")


@pytest.mark.gpu
def test_cuda_raycast_everything_culled(cuda_device):
    """Candidates that all lie beyond the sensor disc (one tile and three tiles), and no candidate at all."""
    rng = np.random.default_rng(9)
    rect, flags = _clutter(rng, 300, lo=R + 3.0, hi=R + 30.0)
    ego = np.array([[0.0, 0.0, 0.2]])
    for bnd in (None, _ring(R + 10.0, 2000)):
        out = _check_frames(ego, rect[None], flags[None], bnd, 360.0, 1024)
        assert (out[0] == np.float32(R)).all() and (out[1] == VO.HIT_NONE).all() and not out[2].any()
    out = _check_frames(ego, np.zeros((1, 0, 5)), np.zeros((1, 0), np.uint8), None, 360.0, 300)
    assert (out[0] == np.float32(R)).all() and (out[1] == VO.HIT_NONE).all()


# ------------------------------------------------------------------------------------------------ angles
def _angle_frame(heading, fov, n_rays, seed):
    """Small boxes straddling ray 0 and every fan boundary (ray 256 k), boxes wholly behind a limited fov, clutter."""
    rng = np.random.default_rng(seed)
    a0, da = (heading - np.pi, 2 * np.pi / n_rays) if fov >= 359.9 else (heading - np.radians(fov) / 2,
                                                                          np.radians(fov) / max(n_rays - 1, 1))
    dirs = [a0] + [a0 + da * 256 * k for k in range(1, (n_rays + 255) // 256)]
    dirs += [heading + np.pi + x for x in (-0.3, 0.0, 0.3)]
    d = 6.0 + 1.5 * np.arange(len(dirs))
    box = np.stack((d * np.cos(dirs), d * np.sin(dirs), rng.uniform(-1, 1, len(dirs)), np.full(len(dirs), 0.4),
                    np.full(len(dirs), 0.25)), -1)
    rect, flags = _clutter(rng, 20)
    return np.concatenate((box, rect)), np.concatenate((np.full(len(box), EX, np.uint8), flags))


@pytest.mark.gpu
@pytest.mark.parametrize("heading", [-np.pi, 0.0, np.pi, 3 * np.pi, -3 * np.pi, 20 * np.pi])
def test_cuda_raycast_angles(heading, cuda_device):
    """Full-circle mode (the wrap clause of the per-fan cull, fan boundaries), the mode switch at 359.9 deg, limited
    fields of view down to 1e-3 deg and 0 (da = 0), one ray in fov mode."""
    for fov in (360.0, 359.9, 359.89, 200.0, 90.0, 1e-3, 0.0):
        for n_rays in ((4096,) if fov >= 359.9 else (4096, 1)):
            rect, flags = _angle_frame(heading, fov, n_rays, seed=int(fov * 10) + n_rays)
            _check_frames(np.array([[0.0, 0.0, heading]]), rect[None], flags[None], _ring(45.0, 64, 3.0), fov, n_rays,
                          what=f"heading {heading} fov {fov} n {n_rays}")


# ------------------------------------------------------------------------------------------------ distances
def _tangent(dist, ang, half=2.0):
    """A border segment whose closest point to the origin lies at ``dist`` in direction ``ang``."""
    c, s = np.cos(ang), np.sin(ang)
    return np.array([dist * c + half * s, dist * s - half * c, dist * c - half * s, dist * s + half * c])


@pytest.mark.gpu
def test_cuda_raycast_distances(cuda_device):
    """Closest points at R -+ 1e-4 (the sensor-disc cull) and hits at t ~ R (t < R strictly on both sides); occluders
    at the ring radii k R / 32 -+ 1e-4 (ring assignment, ring-end exit); occluders 1e-3 .. 1e-7 m from the ego (the
    d2 < 1e-12 branch lists an edge in every fan); an ego inside a box, overlapping, nested, duplicated and zero-size
    boxes."""
    ego = np.array([[0.0, 0.0, 0.4]])
    segs = [_tangent(R + e, a) for e, a in ((-1e-4, 0.1), (1e-4, 0.7), (-1e-6, 1.3), (-1e-5, 1.9))]
    k = np.arange(1, 32)
    rings = [_tangent(kk * R / 32 + e, 2.2 + 0.11 * kk + (0.05 if e > 0 else 0.0), half=0.3)
             for kk in k for e in (-1e-4, 1e-4)]
    near_box = [[R - 1e-4 + 0.5, 0.0, 0.0, 0.5, 0.3]]                        # near face at R - 1e-4 along +x
    rect = np.array(near_box + [[(kk * R / 32 + 1e-4 + 0.2) * np.cos(-1.0 - 0.1 * kk),
                                 (kk * R / 32 + 1e-4 + 0.2) * np.sin(-1.0 - 0.1 * kk), -1.0 - 0.1 * kk, 0.2, 0.15]
                                for kk in k])
    _check_frames(ego, rect[None], np.full((1, len(rect)), EX, np.uint8), np.array(segs + rings), 360.0, 4096,
                  what="R and ring radii")
    tiny = [_tangent(10.0 ** -p, 0.5 + p, half=0.5) for p in range(3, 8)]
    _check_frames(ego, np.zeros((1, 0, 5)), np.zeros((1, 0), np.uint8), np.array(tiny), 360.0, 4096, what="tiny")
    for p in range(3, 8):
        _check_frames(ego, np.zeros((1, 0, 5)), np.zeros((1, 0), np.uint8), tiny[p - 3][None], 360.0, 1024,
                      what=f"tiny 1e-{p}")
        box = np.array([[0.0, 10.0 ** -p + 0.5, 0.0, 1.0, 0.5]])                 # a box side 10^-p from the ego
        _check_frames(ego, box[None], np.ones((1, 1), np.uint8), None, 360.0, 1024, what=f"box 1e-{p}")
    boxes = np.array([[0.5, -0.2, 0.3, 3.0, 2.0],          # contains the ego
                      [0.5, -0.2, 0.3, 1.0, 0.5],          # nested in it, also around the ego
                      [10.0, 3.0, 0.4, 2.0, 1.0], [10.0, 3.0, 0.4, 2.0, 1.0],    # duplicated
                      [11.0, 3.5, -0.3, 2.0, 1.0],         # overlapping them
                      [-8.0, 2.0, 0.0, 0.0, 1.0], [-8.0, -4.0, 0.5, 1.0, 0.0], [4.0, -9.0, 0.0, 0.0, 0.0]])   # zero-size
    flags = np.full((1, len(boxes)), EX, np.uint8)
    _check_frames(ego, boxes[None], flags, None, 360.0, 4096, what="ego inside")
    _check_frames(ego, boxes[None, 2:], flags[:, 2:], None, 360.0, 4096, what="overlapping / zero-size")


# ------------------------------------------------------------------------------------------------ ego on an edge
@pytest.mark.gpu
@pytest.mark.parametrize("n_rays", [16, 4096])
def test_cuda_raycast_ego_on_edge(n_rays, cuda_device):
    """An ego on a box corner or side is blocked at range 0 by exactly the rays that point to the box's side of it
    (``VO.raycast``, the kernel's rule); a zero-width box blocks both sides; a border segment through the ego blocks
    nothing, in either direction.  The far ring must still stop every other ray: a side through the ego can evaluate
    cross(a, e) to -0, and a range of -0 would be the largest key of the warp maximum and end the walk of the warp."""
    ego = np.array([[0.0, 0.0, 0.1]])
    far = f32(_ring(30.0, 50))
    for box in ([2.0, 1.0, 0.0, 2.0, 1.0], [0.0, 1.0, 0.0, 2.0, 1.0], [-2.0, -1.0, 0.0, 2.0, 1.0], [0.0, 0.0, 0.0, 2.0, 0.0],
                [2.0, -1.0, 0.0, 2.0, 1.0], [0.0, -1.0, 0.0, 2.0, 1.0], [-2.0, 1.0, 0.0, 2.0, 1.0]):
        rect = np.array([[box]])
        out = _check_frames(ego, rect, np.ones((1, 1), np.uint8), far, 360.0, n_rays, what=f"box {box}")
        o_rng, o_hit, _ = VO.raycast(ego[0], rect[0], np.ones(1, np.uint8), far, R, 360.0, n_rays)
        assert np.array_equal(out[0][0] == 0, o_rng == 0) and (o_rng == 0).any(), box
        assert np.array_equal(out[1][0][o_rng == 0], o_hit[o_rng == 0])
        assert (out[0][0][o_rng > 0] > 29.0).all(), box
        assert not np.signbit(out[0][0]).any(), box
    seg = np.array([[-5.0, 0.0, 5.0, 0.0], [0.0, 0.0, 3.0, 4.0]])            # through the ego; ending at it
    for bnd in (seg, seg[:, [2, 3, 0, 1]]):
        out = _check_frames(ego, np.zeros((1, 0, 5)), np.zeros((1, 0), np.uint8), np.concatenate((bnd, far)), 360.0,
                            n_rays, what="border through the ego")
        assert (out[0][0] > 29.0).all()


# ------------------------------------------------------------------------------------------------ transparent obstacles
@pytest.mark.gpu
@pytest.mark.parametrize("n_tr", [0, 512, 513, 600])
def test_cuda_raycast_transparent(n_tr, cuda_device):
    """Transparent (bicycle) obstacles: listed in shared memory up to 512, scanned beyond.  One contains the ego, one
    lies wholly behind an occluder, one partly in front of it."""
    rng = np.random.default_rng(n_tr)
    special = np.array([[12.0, 0.0, 0.0, 1.0, 3.0], [0.5, 0.0, 0.0, 1.5, 1.0], [18.0, 0.0, 0.0, 2.0, 1.0],
                        [11.0, 2.5, 0.0, 1.5, 1.0]])  # occluder; bicycles: around the ego, behind it, partly in front
    sflags = np.array([EX, TR, TR, TR], np.uint8)
    if n_tr == 0:
        special, sflags = special[:1], sflags[:1]
    rect, flags = _clutter(rng, n_tr + 100, lo=6.0, hi=48.0)
    rect[:, 3:] *= 0.5
    flags[:max(n_tr - 3, 0)] = TR
    rect, flags = np.concatenate((special, rect)), np.concatenate((sflags, flags))
    assert ((flags & VO.RECT_TRANSPARENT) != 0).sum() == n_tr
    out = _check_frames(np.array([[0.0, 0.0, 0.0]]), rect[None], flags[None], _ring(45.0, 64), 360.0, 2048,
                        what=f"{n_tr} transparent")
    if n_tr:
        assert out[2][0, 1] == 1 and out[2][0, 2] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("n_obst", [65535, 65536])
def test_cuda_raycast_many_obstacles(n_obst, cuda_device):
    """n_obstacles at the limit of the uint16 transparent list (65535) and beyond it (65536: the kernel scans every
    flag), mostly without FO_RECT_EXISTS; existing boxes sit at the end of the list too."""
    rng = np.random.default_rng(n_obst)
    rect = np.zeros((n_obst, 5))
    rect[:, 3:] = 1.0
    flags = np.zeros(n_obst, np.uint8)
    idx = np.concatenate((rng.choice(n_obst - 8, 56, replace=False), np.arange(n_obst - 8, n_obst)))
    rect[idx], flags[idx] = _clutter(rng, len(idx), transparent_every=2)
    _check_frames(np.array([[0.0, 0.0, 1.0]]), rect[None], flags[None], None, 360.0, 256, what=f"O={n_obst}")


@pytest.mark.gpu
def test_cuda_raycast_rays_parallel_to_box_sides(cuda_device):
    """Heading 0, yaw 0 and n_rays a multiple of 4: rays along the axes run parallel to box sides (the slab test's
    parallel branch), some exactly along a bicycle's side."""
    rect = np.array([[10.0, 0.5, 0.0, 1.0, 0.5], [0.0, -8.0, 0.0, 0.5, 1.0], [-6.0, 0.0, 0.0, 1.0, 1.0],
                     [0.0, 15.0, 0.0, 2.0, 1.0], [20.0, 0.0, 0.0, 1.0, 0.5], [-12.0, 1.0, 0.0, 1.0, 1.0]])
    flags = np.array([TR, TR, TR, EX, EX, TR], np.uint8)
    for n in (4, 64, 4096):
        _check_frames(np.array([[0.0, 0.0, 0.0]]), rect[None], flags[None], None, 360.0, n, what=f"n {n}")


@pytest.mark.gpu
def test_cuda_raycast_far_origin(cuda_device):
    """An ego near (1e4, -1e4): the float32 inputs the kernel reads are what the certificate checks."""
    rng = np.random.default_rng(4)
    org = np.array([1e4 + 0.37, -1e4 - 0.61])
    rect, flags = _clutter(rng, 80, transparent_every=5)
    rect[:, :2] += org
    _check_frames(np.array([[org[0], org[1], -2.5]]), rect[None], flags[None], _ring(40.0, 120, 4.0, centre=org), 360.0,
                  4096, what="far origin")


# ------------------------------------------------------------------------------------------------ frames, C-ABI
@pytest.mark.gpu
def test_cuda_raycast_frames_above_grid_limit(cuda_device):
    """65537 frames: raycast_frames splits them at the 65535-frame grid limit; the frames around the split equal their
    single-frame casts."""
    F = 65537
    ego = np.zeros((F, 3))
    ego[:, 2] = np.linspace(-3.0, 3.0, F)
    base = np.array([[8.0, 1.0, 0.2, 1.0, 0.5], [-5.0, -3.0, 1.0, 2.0, 1.0], [1.0, 9.0, 0.0, 0.5, 0.5]])
    rect = np.repeat(base[None], F, 0)
    rect[:, :, 0] += np.linspace(0.0, 1.0, F)[:, None]
    flags = np.full((F, 3), EX, np.uint8)
    flags[:, 2] = TR
    ego, rect = f32(ego), f32(rect)
    out = cast(ego, rect, flags, None, R, 360.0, 32)
    for f in (0, 65533, 65534, 65535, 65536):
        one = cast(ego[f:f + 1], rect[f:f + 1], flags[f:f + 1], None, R, 360.0, 32)
        assert_same_or_tied(one, tuple(o[f:f + 1] for o in out), lambda _: (ego[f], rect[f], flags[f], None), R, 360.0,
                            32, what=f"frame {f}")
        certify(one, 0, ego[f], rect[f], flags[f], None, R, 360.0, 32)


def test_raycast_capi_rejects_65536_frames():
    """A direct call with 65536 frames returns FO_ERR_UNSUPPORTED before it touches a device."""
    from frenetix_occlusion_b200 import _lib as L
    buf = (C.c_float * 16)()
    v = L.FoVisibilityArgs()
    v.n_frames, v.n_rays, v.sensor_radius, v.sensor_angle_deg = 65536, 8, 50.0, 360.0
    v.ego, v.range, v.hit = (C.cast(buf, C.c_void_p),) * 3
    assert L.lib.fo_visibility_raycast(C.byref(v), None) == -2
    assert b"65535" in L.lib.fo_last_error()


@pytest.mark.gpu
def test_cuda_raycast_capi_without_visible(cuda_device):
    """visible = NULL: range and hit equal the call that writes visible."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    ego, rect, flags, bnd = _pool()
    n = 1024
    ref = cast(ego, rect, flags, bnd, R, 360.0, n)
    dev = cuda_device
    d_ego, d_rect = torch.from_numpy(ego.astype(np.float32)).to(dev), torch.from_numpy(rect.astype(np.float32)).to(dev)
    d_flags, d_bnd = torch.from_numpy(flags).to(dev), torch.from_numpy(bnd.astype(np.float32)).to(dev)
    rng_, hit = torch.full((4, n), float("nan"), device=dev), torch.full((4, n), 99, dtype=torch.int32, device=dev)
    a = L.FoVisibilityArgs()
    a.n_frames, a.n_rays, a.n_obstacles, a.n_boundary = 4, n, rect.shape[1], len(bnd)
    a.ego, a.rect, a.rect_flags, a.boundary = d_ego.data_ptr(), d_rect.data_ptr(), d_flags.data_ptr(), d_bnd.data_ptr()
    a.sensor_radius, a.sensor_angle_deg = R, 360.0
    a.range, a.hit, a.visible = rng_.data_ptr(), hit.data_ptr(), None
    L.check(L.lib.fo_visibility_raycast(C.byref(a), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "raycast")
    torch.cuda.synchronize()
    out = (rng_.cpu().numpy(), hit.cpu().numpy(), ref[2])
    assert_same_or_tied(ref, out, lambda f: (ego[f], rect[f], flags[f], bnd), R, 360.0, n, what="visible NULL")


# ------------------------------------------------------------------------------------------------ invariances
@pytest.mark.gpu
def test_cuda_raycast_invariances(cuda_device):
    """Reversing every border segment changes nothing, splitting a border segment at its midpoint changes nothing but
    certified ties, permuting obstacles permutes owners and visible."""
    ego, rect, flags, bnd = _pool()
    n = 4096
    frame = lambda f: (ego[f], rect[f], flags[f], bnd)
    ref = cast(ego, rect, flags, bnd, R, 360.0, n)
    rev = cast(ego, rect, flags, bnd[:, [2, 3, 0, 1]], R, 360.0, n)
    assert_same_or_tied(ref, rev, frame, R, 360.0, n, what="reversed", ulp=None)
    mid = f32((bnd[:, :2] + bnd[:, 2:]) / 2)
    split = np.concatenate((np.concatenate((bnd[:, :2], mid), 1), np.concatenate((mid, bnd[:, 2:]), 1)))
    spl = cast(ego, rect, flags, split, R, 360.0, n)
    for f in range(4):
        certify(spl, f, ego[f], rect[f], flags[f], split, R, 360.0, n, what="split")
    assert_same_or_tied(ref, spl, frame, R, 360.0, n, what="split", ulp=None)
    perm = np.random.default_rng(2).permutation(rect.shape[1])
    p = cast(ego, rect[:, perm], flags[:, perm], bnd, R, 360.0, n)
    mapped = np.where(p[1] >= 0, perm[np.maximum(p[1], 0)], p[1])
    assert np.array_equal(p[2], ref[2][:, perm])
    assert_same_or_tied(ref, (p[0], mapped, p[2][:, np.argsort(perm)]), frame, R, 360.0, n, what="permuted")


# ------------------------------------------------------------------------------------------------ fo_rollout_cv
def _cv_agents():
    phi = np.array([0.0, np.pi / 2, -np.pi / 2, np.pi, -np.pi, 0.3, -2.1, 1.0])
    v = np.array([1.4, 2.0, 0.0, 3.3, 1.1, 0.0, 7.9, 12.0])
    x0 = np.array([0.0, 1e5 + 0.123, -1e5 - 0.77, 12.5, 1e5, -3.0, 99999.9, 5.5])
    y0 = np.array([0.0, -1e5 + 0.5, 3.0, 1e5 - 0.01, 7.0, -1e5, 0.25, -2.0])
    return x0, y0, v, phi


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [0.05, 0.2, 0.25])
@pytest.mark.parametrize("var0,var_factor", [(0.1, 1.0), (0.1, 0.9), (0.37, 1.05)])
def test_cuda_rollout_cv_edges(dt, var0, var_factor, cuda_device):
    """Bit-exact against VO.rollout_cv: time steps, variance factors 1.0 and 0.9 and a non-default var0, v = 0,
    headings 0, +-pi/2, +-pi, starts near 1e5 m, and one state (horizon 0)."""
    import torch
    from frenetix_occlusion_b200.prediction import rollout_cv
    x0, y0, v, phi = _cv_agents()
    for horizon in (5.0, 0.0):
        g = rollout_cv(x0, y0, v, phi, dt, horizon, var0=var0, var_factor=var_factor)
        torch.cuda.synchronize()
        o = VO.rollout_cv(x0, y0, v, phi, dt, horizon, var0=var0, var_factor=var_factor)
        assert o["x"].shape[1] == (1 if horizon == 0.0 else int(horizon / dt) + 1)
        for key in ("x", "y", "yaw", "v", "var"):
            assert np.array_equal(g[key].cpu().numpy(), o[key].astype(np.float32)), (key, horizon)


@pytest.mark.gpu
def test_cuda_rollout_cv_padding(cuda_device):
    """Direct C-ABI call with t_stride = n_states + 5 into NaN-filled outputs: the padding is written with zeros and the
    rows equal the oracle; var_y equals var_x."""
    import torch
    from frenetix_occlusion_b200 import _lib as L
    x0, y0, v, phi = _cv_agents()
    A, dt, horizon = len(x0), 0.1, 3.0
    T = int(horizon / dt) + 1
    S = T + 5
    dev = cuda_device
    inp = torch.from_numpy(np.stack([x0, y0, v, phi])).to(dev)
    out = torch.full((6, A, S), float("nan"), dtype=torch.float32, device=dev)
    a = L.FoRolloutCvArgs()
    a.n_agents, a.n_states, a.t_stride, a.dt, a.var0, a.var_factor = A, T, S, dt, 0.1, 1.05
    a.x0, a.y0, a.v, a.phi = [inp[i].data_ptr() for i in range(4)]
    a.x, a.y, a.yaw, a.vel, a.var_x, a.var_y = [out[i].data_ptr() for i in range(6)]
    L.check(L.lib.fo_rollout_cv(C.byref(a), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "fo_rollout_cv")
    torch.cuda.synchronize()
    g = out.cpu().numpy()
    assert np.array_equal(g[:, :, T:], np.zeros((6, A, 5), np.float32))
    o = VO.rollout_cv(x0, y0, v, phi, dt, horizon)
    for i, key in enumerate(("x", "y", "yaw", "v", "var")):
        assert np.array_equal(g[i, :, :T], o[key].astype(np.float32)), key
    assert np.array_equal(g[5], g[4])
