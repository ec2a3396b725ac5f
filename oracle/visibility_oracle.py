"""Oracle for stage 1 (sensor visibility) and stage 2 (constant-velocity rollout).  TEST INFRASTRUCTURE.

PARITY UNPINNED at the polygon level: the reference builds its visible area with shapely/GEOS
boolean operations (``sensor_model.py:103-193``), which cannot be installed here, and ships no test
vectors.  Two restatements are kept instead:

* ``reference_point_visible``  -- the reference's own construction evaluated point-wise, polygon-library
  free: a point is visible iff it lies in the sensor sector, in none of the per-border-edge shadow
  quads ``[v1, v2, v2+100(v2-ego), v1+100(v1-ego)]`` (``sensor_model.py:137-155``,
  ``helper_functions.py:79-96``) and in none of the per-obstacle shadows built from the corner pair
  with the largest subtended angle (``helper_functions.py:139-176``) united with the obstacle itself
  (``sensor_model.py:174-191``); bicycles cast no shadow (``sensor_model.py:177``).
* ``raycast`` -- float64 brute-force restatement of the ray-cast formulation the CUDA kernel uses
  (first hit of every ray of the fan), bit-for-bit the same angle convention and hit rule.  The
  tests check ``raycast`` == ``reference_point_visible`` up to the angular resolution of the fan, and
  hold every ray and visible flag of the kernel to ``certify_raycast`` (float64, tolerance
  5e-5 + 1e-5 rho m); ``raycast_f32`` restates the kernel's float32 arithmetic so the certificate
  itself can be tested on the CPU.
"""
from __future__ import annotations

import numpy as np

HIT_NONE, HIT_BOUNDARY = -1, -2
RECT_EXISTS, RECT_TRANSPARENT = 1, 2


def ray_angles(heading: float, fov_deg: float, n_rays: int) -> np.ndarray:
    if fov_deg >= 359.9:                                   # sensor_model.py:119-120 (full disc)
        return heading - np.pi + 2.0 * np.pi * np.arange(n_rays) / n_rays
    fov = np.radians(fov_deg)
    return heading - 0.5 * fov + (fov / max(n_rays - 1, 1)) * np.arange(n_rays)


def rect_corners(rect: np.ndarray) -> np.ndarray:
    """[O,5] (cx, cy, yaw, hl, hw) -> [O,4,2] corner ring in commonroad ``Rectangle.vertices`` order,
    rotated and translated as ``hf.calc_corner_points`` does (helper_functions.py:99-112)."""
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    sx = np.array([-1.0, -1.0, 1.0, 1.0])
    sy = np.array([-1.0, 1.0, 1.0, -1.0])
    lx = sx[None] * rect[:, 3:4]
    ly = sy[None] * rect[:, 4:5]
    c, s = np.cos(rect[:, 2:3]), np.sin(rect[:, 2:3])
    return np.stack((rect[:, 0:1] + lx * c - ly * s, rect[:, 1:2] + lx * s + ly * c), -1)


def _edges(ego_xy, rect, flags, boundary):
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    flags = np.asarray(flags).reshape(-1)
    segs, owner = [], []
    cor = rect_corners(rect)
    for o in range(len(rect)):
        if (flags[o] & RECT_EXISTS) and not (flags[o] & RECT_TRANSPARENT):
            for e in range(4):
                segs.append(np.concatenate((cor[o, e], cor[o, (e + 1) % 4])))
                owner.append(o)
    if boundary is not None and len(boundary):
        for b in np.asarray(boundary, dtype=np.float64).reshape(-1, 4):
            segs.append(b)
            owner.append(HIT_BOUNDARY)
    segs = np.asarray(segs, dtype=np.float64).reshape(-1, 4)
    segs = segs - np.tile(np.asarray(ego_xy, dtype=np.float64), 2)
    return segs, np.asarray(owner, dtype=np.int64)


def _oriented(segs, owner):
    """The edges as the kernel stages them: a border segment whose line passes exactly through the ego (cross(a, e)
    == 0) is dropped -- it could only block at range 0, and only on the side its listed direction happens to face --
    and every other edge is oriented so that cross(a, e) >= 0 (an edge with cross(a, e) == 0 keeps its listed
    direction: a rectangle side through the ego blocks the rays that point to the box's side of it).
    Returns (a [E,2], e [E,2], tn [E], owner [E])."""
    a, e = segs[:, :2].copy(), segs[:, 2:] - segs[:, :2]
    tn = a[:, 0] * e[:, 1] - a[:, 1] * e[:, 0]
    keep = ~((owner == HIT_BOUNDARY) & (tn == 0))
    a, e, tn, owner = a[keep], e[keep], tn[keep], owner[keep]
    fl = tn < 0
    a[fl] += e[fl]
    e[fl], tn[fl] = -e[fl], -tn[fl]
    return a, e, tn, owner


def _first_hits(a, e, tn, c, s, sensor_radius):
    """Float64 first hit of rays (c, s) [N,1] on oriented edges: hit iff D = cross(d, e) > 0, 0 <= cross(a, d) <= D
    and t = tn / D < sensor_radius.  Returns (t [N], edge index [N]); t = inf where nothing is hit."""
    n = len(c)
    if not len(a):
        return np.full(n, np.inf), np.zeros(n, dtype=np.int64)
    D = c * e[None, :, 1] - s * e[None, :, 0]
    un = a[None, :, 0] * s - a[None, :, 1] * c
    with np.errstate(divide="ignore", invalid="ignore"):
        t = tn[None] / D
    t = np.where((D > 0) & (un >= 0) & (un <= D) & (t < sensor_radius), t, np.inf)
    j = t.argmin(1)
    return t[np.arange(n), j], j


def _box_frame(rect, ego_xy, c, s):
    """Rays (c, s) [N] in the frames of boxes rect [T,5]: origin (ox, oy) [T] and direction (dx, dy) [N,T]."""
    cx, cy = rect[:, 0] - ego_xy[0], rect[:, 1] - ego_xy[1]
    cs, sn = np.cos(rect[:, 2]), np.sin(rect[:, 2])
    ox, oy = -(cx * cs + cy * sn), -(-cx * sn + cy * cs)
    return ox, oy, c[:, None] * cs + s[:, None] * sn, -c[:, None] * sn + s[:, None] * cs


def raycast(ego, rect, flags, boundary, sensor_radius, fov_deg, n_rays):
    """First-hit range / hit id per ray and per-obstacle visibility for ONE frame (float64).  Edges are staged as the
    kernel stages them (``_oriented``): an ego standing on a rectangle side is blocked at range 0 exactly by the rays
    that point to the box's side of it (at a corner: of either side), and a border segment through the ego blocks nothing."""
    ego = np.asarray(ego, dtype=np.float64)
    ang = ray_angles(ego[2], fov_deg, n_rays)
    c, s = np.cos(ang)[:, None], np.sin(ang)[:, None]
    segs, owner = _edges(ego[:2], rect, flags, boundary)
    a, e, tn, owner = _oriented(segs, owner)
    tb, j = _first_hits(a, e, tn, c, s, sensor_radius)
    better = tb < sensor_radius
    rng = np.where(better, tb, float(sensor_radius))
    hit = np.where(better, owner[j] if len(owner) else HIT_NONE, HIT_NONE).astype(np.int64)
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    flags = np.asarray(flags).reshape(-1)
    visible = np.zeros(len(rect), dtype=np.uint8)
    for o in np.unique(hit[hit >= 0]):
        visible[o] = 1
    for o in range(len(rect)):                             # transparent obstacles: slab test up to the first hit
        if (flags[o] & RECT_EXISTS) and (flags[o] & RECT_TRANSPARENT):
            hl, hw = rect[o, 3], rect[o, 4]
            ox, oy, dx, dy = _box_frame(rect[o:o + 1], ego, c[:, 0], s[:, 0])
            dx, dy = dx[:, 0], dy[:, 0]
            with np.errstate(divide="ignore", invalid="ignore"):
                tx0, tx1 = (-hl - ox) / dx, (hl - ox) / dx
                ty0, ty1 = (-hw - oy) / dy, (hw - oy) / dy
            t0 = np.maximum(np.minimum(tx0, tx1), np.minimum(ty0, ty1))
            t1 = np.minimum(np.maximum(tx0, tx1), np.maximum(ty0, ty1))
            if np.any((np.maximum(t0, 0.0) <= np.minimum(t1, rng))):
                visible[o] = 1
    return rng, hit, visible


def raycast_f32(ego, rect, flags, boundary, sensor_radius, fov_deg, n_rays):
    """numpy float32 restatement of the kernel's arithmetic for ONE frame, without its culls and sort: float32 ray
    angles a0 + da r, corners from float32 sin / cos of the yaw, the staging orientation flip (border segments with
    cross(a, e) == 0 dropped), the division-free hit test D > 0, 0 <= un <= D, tn < best D, and the transparent slab
    test up to the first opaque hit.  Returns (range f32 [N], hit [N], visible u8 [O])."""
    f32 = np.float32
    ego = np.asarray(ego, dtype=f32)
    rect = np.asarray(rect, dtype=f32).reshape(-1, 5)
    flags = np.asarray(flags, dtype=np.uint8).reshape(-1)
    R, pi = f32(sensor_radius), f32(np.pi)
    if fov_deg >= 359.9:
        a0, da = f32(ego[2] - pi), f32(f32(2.0) * pi / f32(n_rays))
    else:
        fov = f32(f32(fov_deg) * f32(pi / f32(180.0)))
        a0 = f32(ego[2] - f32(0.5) * fov)
        da = f32(fov / f32(n_rays - 1)) if n_rays > 1 else f32(0.0)
    th = a0 + da * np.arange(n_rays, dtype=f32)
    c, s = np.cos(th)[:, None], np.sin(th)[:, None]
    rel = rect[:, :2] - ego[:2]
    sn, cs = np.sin(rect[:, 2]), np.cos(rect[:, 2])
    sx = np.array([-1, -1, 1, 1], dtype=f32)
    sy = np.array([-1, 1, 1, -1], dtype=f32)
    hl, hw = rect[:, 3:4], rect[:, 4:5]
    px = rel[:, 0:1] + sx * hl * cs[:, None] - sy * hw * sn[:, None]       # [O, 4] corners, ego frame
    py = rel[:, 1:2] + sx * hl * sn[:, None] + sy * hw * cs[:, None]
    opaque = (flags & RECT_EXISTS).astype(bool) & ~(flags & RECT_TRANSPARENT).astype(bool)
    nxt = [1, 2, 3, 0]
    g = np.stack((px, py, px[:, nxt], py[:, nxt]), -1)[opaque].reshape(-1, 4)
    own = np.repeat(np.flatnonzero(opaque), 4)
    if boundary is not None and len(boundary):
        b = np.asarray(boundary, dtype=f32).reshape(-1, 4) - np.tile(ego[:2], 2)
        g = np.concatenate((g, b))
        own = np.concatenate((own, np.full(len(b), HIT_BOUNDARY)))
    ax, ay = g[:, 0].copy(), g[:, 1].copy()
    ex, ey = g[:, 2] - ax, g[:, 3] - ay
    tn = ax * ey - ay * ex
    keep = ~((own == HIT_BOUNDARY) & (tn == 0))
    ax, ay, ex, ey, tn, own, g = ax[keep], ay[keep], ex[keep], ey[keep], tn[keep], own[keep], g[keep]
    fl = tn < 0
    ax[fl], ay[fl] = g[fl, 2], g[fl, 3]
    ex[fl], ey[fl], tn[fl] = -ex[fl], -ey[fl], -tn[fl]
    tn = np.abs(tn)                                        # +0 for an edge through the ego, as the kernel stages it
    D = c * ey - s * ex
    un = ax * s - ay * c
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where((D > 0) & (un >= 0) & (un <= D) & (tn < R * D), tn / D, f32(np.inf)).astype(f32)
    if len(own):
        j = t.argmin(1)
        tb = t[np.arange(n_rays), j]
    else:
        j, tb = np.zeros(n_rays, dtype=np.int64), np.full(n_rays, np.inf, dtype=f32)
    hitp = np.isfinite(tb)
    rng = np.where(hitp, tb, R).astype(f32)
    hit = np.where(hitp, own[j] if len(own) else HIT_NONE, HIT_NONE).astype(np.int64)
    visible = np.zeros(len(rect), dtype=np.uint8)
    visible[np.unique(hit[hit >= 0])] = 1
    for o in np.flatnonzero((flags & RECT_EXISTS).astype(bool) & (flags & RECT_TRANSPARENT).astype(bool)):
        ox, oy = -(rel[o, 0] * cs[o] + rel[o, 1] * sn[o]), -(-rel[o, 0] * sn[o] + rel[o, 1] * cs[o])
        dx, dy = c[:, 0] * cs[o] + s[:, 0] * sn[o], -c[:, 0] * sn[o] + s[:, 0] * cs[o]
        t0, t1, ok = np.zeros(n_rays, f32), rng.copy(), np.ones(n_rays, bool)
        for dd, oo, h in ((dx, ox, rect[o, 3]), (dy, oy, rect[o, 4])):
            par = np.abs(dd) <= f32(1e-12)
            with np.errstate(divide="ignore", invalid="ignore"):
                ta, tb2 = (-h - oo) / dd, (h - oo) / dd
            t0 = np.where(par, t0, np.maximum(t0, np.minimum(ta, tb2)))
            t1 = np.where(par, t1, np.minimum(t1, np.maximum(ta, tb2)))
            ok &= ~(par & (np.abs(oo) > h))
        if np.any(ok & (t0 <= t1)):
            visible[o] = 1
    return rng, hit, visible


# ------------------------------------------------------------------------------------------------
CERT_D0, CERT_D1 = 5e-5, 1e-5         # certificate tolerance delta(rho) = CERT_D0 + CERT_D1 rho  [m]


def _seg_seg_dist(p0, p1, a, b):
    """Distance between segment p0 -> p1 and segments a -> b [E,2] (float64)."""
    def pt_seg(p, q0, q1):
        e = q1 - q0
        l2 = (e * e).sum(-1)
        u = np.clip(((p - q0) * e).sum(-1) / np.maximum(l2, 1e-300), 0.0, 1.0)
        return np.hypot(*(q0 + u[..., None] * e - p).T)

    def cr(o, x, y):
        return (x[..., 0] - o[..., 0]) * (y[..., 1] - o[..., 1]) - (x[..., 1] - o[..., 1]) * (y[..., 0] - o[..., 0])

    p0, p1 = np.broadcast_to(p0, a.shape), np.broadcast_to(p1, a.shape)
    cross = (cr(p0, p1, a) * cr(p0, p1, b) < 0) & (cr(a, b, p0) * cr(a, b, p1) < 0)
    dmin = np.minimum(np.minimum(pt_seg(p0, a, b), pt_seg(p1, a, b)), np.minimum(pt_seg(a, p0, p1), pt_seg(b, p0, p1)))
    return np.where(cross, 0.0, dmin)


def _segment_meets_box(L, c, s, rect, ego_xy, grow):
    """Does the sight segment [0, L d] (L [N], d = (c, s) [N]) meet box rect [T,5] with half extents grown by ``grow``
    ([N], negative: shrunk)?  Float64 slab test; [N, T] bool."""
    ox, oy, dx, dy = _box_frame(rect, ego_xy, c, s)
    t0, t1 = np.zeros(dx.shape), np.broadcast_to(L[:, None], dx.shape).copy()
    ok = np.ones(dx.shape, bool)
    for dd, oo, h in ((dx, ox, rect[:, 3]), (dy, oy, rect[:, 4])):
        h = h[None] + grow[:, None]
        ok &= h >= 0
        par = dd == 0
        with np.errstate(divide="ignore", invalid="ignore"):
            ta, tb = (-h - oo) / dd, (h - oo) / dd
        t0 = np.where(par, t0, np.maximum(t0, np.minimum(ta, tb)))
        t1 = np.where(par, t1, np.minimum(t1, np.maximum(ta, tb)))
        ok &= ~(par & (np.abs(oo) > h))
    return ok & (t0 <= t1)


def certify_raycast(range_, hit, visible, ego, rect, flags, boundary, sensor_radius, fov_deg, n_rays,
                    d0=CERT_D0, d1=CERT_D1, rays=None, chunk=256):
    """Certify a ray cast of ONE frame in float64, ray by ray, with tolerance delta(rho) = d0 + d1 rho [m].  Ray r has
    the float64 direction d at its nominal angle (``ray_angles``) and the answer (rho, h); P = rho d.

    (A) the reported hit is real: h == HIT_NONE and rho == float32(R), or some edge of owner h lies within delta of P;
    (B) no nearer hit was missed: no edge crosses the sight segment [0, P] robustly -- its end points on opposite
        sides of the ray line and 0 and P on opposite sides of its line, each at least delta away.  The margins are
        perpendicular, so grazing rays, whose range is ill-conditioned, pass;
    (V) ``visible`` (may be None): every hit owner is visible; an opaque visible obstacle is some ray's hit; a
        transparent visible obstacle meets some sight segment [0, (rho + delta) d] within delta.  An invisible opaque
        obstacle is no ray's robust float64 first hit (crossed robustly, before R - delta, with no other owner's edge
        within delta of the sight segment up to delta beyond it); an invisible transparent obstacle, shrunk by delta,
        meets no sight segment [0, (rho - delta) d].

    Inputs are the kernel's (float32 numbers in float64 arrays).  ``rays``: check only these rays (``range_`` and
    ``hit`` then hold just their answers, and ``visible`` must be None).  Returns a dict: ``ray_ok`` bool [N], ``ray_reason``
    list of str ('' where ok), ``vis_ok`` bool [O], ``vis_reason`` list of str, ``n_fail`` = failed rays + obstacles."""
    ego = np.asarray(ego, dtype=np.float64)
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    flags = np.asarray(flags).reshape(-1)
    rho = np.asarray(range_, dtype=np.float64).reshape(-1)
    hit = np.asarray(hit).astype(np.int64).reshape(-1)
    R = float(sensor_radius)
    R32 = float(np.float32(R))
    ang = ray_angles(float(ego[2]), fov_deg, n_rays)
    if rays is not None:
        assert visible is None, "visibility is certified over all rays of the frame"
        ang = ang[np.asarray(rays, dtype=np.int64)]
        n_rays = len(ang)
    c, s = np.cos(ang), np.sin(ang)
    delta = d0 + d1 * rho
    P = rho[:, None] * np.stack((c, s), -1)
    segs, owner = _edges(ego[:2], rect, flags, boundary)
    a, b = segs[:, :2], segs[:, 2:]
    e = b - a
    le = np.hypot(e[:, 0], e[:, 1])
    ray_ok = np.ones(n_rays, bool)
    reason = [""] * n_rays
    for r in np.flatnonzero(~np.isfinite(rho) | (rho < 0) | (rho > R32)):
        ray_ok[r], reason[r] = False, f"range {rho[r]!r} outside [0, R]"
    for r in np.flatnonzero(ray_ok & (hit == HIT_NONE) & (rho != R32)):
        ray_ok[r], reason[r] = False, f"A: no hit but range {rho[r]!r} != R"
    for r in np.flatnonzero(ray_ok & (hit != HIT_NONE) & ~np.isin(hit, owner)):
        ray_ok[r], reason[r] = False, f"A: owner {hit[r]} has no edge"
    for r0 in range(0, n_rays, chunk):
        sl = slice(r0, min(n_rays, r0 + chunk))
        if not len(segs):
            break
        Pc, dl = P[sl], delta[sl, None]
        # (A)
        u = np.clip(((Pc[:, None] - a) * e).sum(-1) / np.maximum(le * le, 1e-300), 0.0, 1.0)
        dist = np.hypot(*(a + u[..., None] * e - Pc[:, None]).transpose(2, 0, 1))
        near = ((dist <= dl) & (owner[None] == hit[sl, None])).any(1)
        for k in np.flatnonzero(~near & (hit[sl] != HIT_NONE) & ray_ok[sl]):
            r = r0 + k
            ray_ok[r], reason[r] = False, f"A: no edge of owner {hit[r]} within {delta[r]:.2e} of the hit at {rho[r]!r}"
        # (B)
        cc, ss = c[sl, None], s[sl, None]
        ca = cc * a[None, :, 1] - ss * a[None, :, 0]
        cb = cc * b[None, :, 1] - ss * b[None, :, 0]
        with np.errstate(divide="ignore", invalid="ignore"):
            s0 = (e[None, :, 0] * -a[None, :, 1] - e[None, :, 1] * -a[None, :, 0]) / le
            s1 = (e[None, :, 0] * (Pc[:, None, 1] - a[None, :, 1]) - e[None, :, 1] * (Pc[:, None, 0] - a[None, :, 0])) / le
        robust = ((ca * cb < 0) & (np.abs(ca) >= dl) & (np.abs(cb) >= dl)
                  & (s0 * s1 < 0) & (np.abs(s0) >= dl) & (np.abs(s1) >= dl))
        for k in np.flatnonzero(robust.any(1) & ray_ok[sl]):
            r = r0 + k
            j = int(np.flatnonzero(robust[k])[0])
            ray_ok[r], reason[r] = False, f"B: edge {j} of owner {owner[j]} crosses the sight segment before {rho[r]!r}"
    vis_ok = np.ones(len(rect), bool)
    vis_reason = [""] * len(rect)
    if visible is not None:
        visible = np.asarray(visible).reshape(-1)
        exists = (flags & RECT_EXISTS).astype(bool)
        transp = exists & (flags & RECT_TRANSPARENT).astype(bool)
        opaque = exists & ~transp
        hit_owners = np.unique(hit[hit >= 0])
        for o in hit_owners[visible[hit_owners] == 0]:
            vis_ok[o], vis_reason[o] = False, "V: some ray hits it but visible = 0"
        for o in np.flatnonzero((visible != 0) & ~exists):
            vis_ok[o], vis_reason[o] = False, "V: visible but does not exist"
        for o in np.flatnonzero((visible != 0) & opaque & ~np.isin(np.arange(len(rect)), hit_owners)):
            vis_ok[o], vis_reason[o] = False, "V: opaque, visible, but no ray hits it"
        tr = np.flatnonzero(transp)
        if len(tr):
            for o_set, L, grow, want in ((tr[visible[tr] != 0], rho + delta, delta, True),
                                          (tr[visible[tr] == 0], rho - delta, -delta, False)):
                if not len(o_set):
                    continue
                meet = _segment_meets_box(np.maximum(L, 0.0), c, s, rect[o_set], ego, grow).any(0)
                for k in np.flatnonzero(meet != want):
                    o = o_set[k]
                    vis_ok[o] = False
                    vis_reason[o] = ("V: transparent, visible, but no sight segment comes within delta" if want else
                                     "V: transparent, visible = 0, but a sight segment crosses it robustly")
        hidden = opaque & (visible == 0)
        if hidden.any() and len(segs):
            oa, oe, otn, oown = _oriented(segs, owner)
            t64, j64 = _first_hits(oa, oe, otn, c[:, None], s[:, None], R)
            cand = np.flatnonzero(np.isfinite(t64) & (oown[j64] >= 0))
            cand = cand[hidden[oown[j64[cand]]]]
            for r in cand:
                o, j, t = int(oown[j64[r]]), int(j64[r]), float(t64[r])
                dl = d0 + d1 * t
                d = np.array([c[r], s[r]])
                pa, pb = oa[j], oa[j] + oe[j]
                if not (t < R - dl and abs(d[0] * pa[1] - d[1] * pa[0]) >= dl and abs(d[0] * pb[1] - d[1] * pb[0]) >= dl
                        and otn[j] / np.hypot(*oe[j]) >= dl):
                    continue
                other = owner != o
                if other.any() and (_seg_seg_dist(np.zeros(2), (t + dl) * d, a[other], b[other]) <= dl).any():
                    continue
                vis_ok[o], vis_reason[o] = False, f"V: visible = 0 but ray {r} sees it robustly at {t:.6f}"
    return {"ray_ok": ray_ok, "ray_reason": reason, "vis_ok": vis_ok, "vis_reason": vis_reason,
            "n_fail": int((~ray_ok).sum() + (~vis_ok).sum())}


def certificate_failures(cert, limit=8):
    """Readable summary of a ``certify_raycast`` result's failures (for assertion messages)."""
    out = [f"ray {r}: {cert['ray_reason'][r]}" for r in np.flatnonzero(~cert["ray_ok"])[:limit]]
    out += [f"obstacle {o}: {cert['vis_reason'][o]}" for o in np.flatnonzero(~cert["vis_ok"])[:limit]]
    return f"{cert['n_fail']} failures: " + "; ".join(out)


# ------------------------------------------------------------------------------------------------
def _angle_between(v1, v2):
    v1 = v1 / np.linalg.norm(v1)
    v2 = v2 / np.linalg.norm(v2)
    return np.arccos(np.clip(np.dot(v1, v2), -1.0, 1.0))


def identify_projection_points(ego_xy, corner_points):
    """helper_functions.py:157-176: the corner pair with the largest subtended angle (first maximum)."""
    max_angle = 0
    ret = (corner_points[0], corner_points[0])
    for p1 in corner_points:
        for p2 in corner_points:
            a = _angle_between(p1 - ego_xy, p2 - ego_xy)
            if a > max_angle:
                max_angle = a
                ret = (p1, p2)
    return ret


def _in_convex_quad(P, quad):
    """Closed point-in-convex-polygon test for points [M,2]; orientation independent."""
    q = np.asarray(quad, dtype=np.float64)
    e = np.roll(q, -1, axis=0) - q
    rel = P[:, None, :] - q[None]
    cr = e[None, :, 0] * rel[..., 1] - e[None, :, 1] * rel[..., 0]
    return np.all(cr >= 0, 1) | np.all(cr <= 0, 1)


def reference_point_visible(P, ego, rect, flags, boundary, sensor_radius, fov_deg):
    """Point-wise evaluation of the reference's visible-area construction (see module docstring).
    ``boundary``: [B,4] consecutive exterior-vertex pairs (x1,y1,x2,y2) of road ∩ sector."""
    P = np.asarray(P, dtype=np.float64).reshape(-1, 2)
    ego = np.asarray(ego, dtype=np.float64)
    e = ego[:2]
    d = P - e
    r = np.hypot(d[:, 0], d[:, 1])
    vis = r <= sensor_radius
    if fov_deg < 359.9:                                    # sensor_model.py:201-209 sector
        rel = (np.arctan2(d[:, 1], d[:, 0]) - ego[2] + np.pi) % (2 * np.pi) - np.pi
        vis &= np.abs(rel) <= np.radians(fov_deg) / 2
    if boundary is not None:
        for b in np.asarray(boundary, dtype=np.float64).reshape(-1, 4):
            v1, v2 = b[:2], b[2:]
            quad = [v1, v2, v2 + 100 * (v2 - e), v1 + 100 * (v1 - e)]   # helper_functions.py:90-94
            vis &= ~_in_convex_quad(P, quad)
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    cor = rect_corners(rect)
    for o in range(len(rect)):
        if not (flags[o] & RECT_EXISTS) or (flags[o] & RECT_TRANSPARENT):   # sensor_model.py:177
            continue
        c1, c2 = identify_projection_points(e, cor[o])
        u1 = (c1 - e) / np.linalg.norm(c1 - e)
        u2 = (c2 - e) / np.linalg.norm(c2 - e)
        quad = [c1, c2, c2 + u2 * 100, c1 + u1 * 100]                    # helper_functions.py:143-148
        vis &= ~_in_convex_quad(P, quad)
        vis &= ~_in_convex_quad(P, cor[o])                                # obstacle polygon itself
    return vis


# ------------------------------------------------------------------------------------------------
def rollout_cv(x0, y0, v, phi, dt, horizon, var0=0.1, var_factor=1.05):
    """Pedestrian constant-velocity prediction, float64, exactly the reference's arithmetic
    (agent.py:487-503, 520-536, 260-280).  Returns dict of [A,T] arrays."""
    x0, y0, v, phi = (np.atleast_1d(np.asarray(a, dtype=np.float64)) for a in (x0, y0, v, phi))
    n = int(horizon / dt) + 1                                              # agent.py:496
    vx = np.array([round(float(a), 3) for a in v * np.cos(phi)])          # agent.py:492
    vy = np.array([round(float(a), 3) for a in v * np.sin(phi)])          # agent.py:493
    t = np.arange(n)[None, :] * dt                                         # agent.py:499
    k = np.arange(n)
    return {"x": x0[:, None] + t * vx[:, None], "y": y0[:, None] + t * vy[:, None],
            "yaw": np.repeat(phi[:, None], n, 1), "v": np.repeat(v[:, None], n, 1),
            "var": np.repeat((var0 * np.power(var_factor, k))[None], len(v), 0)}


MIN_CHORD = 1e-3          # [m] fo_rollout.cu kMinChord


def rollout_path(path, x0, y0, v0, dt, horizon, t1=3.0, var0=0.1, var_factor=1.05):
    """float64 restatement of the path-following vehicle rollout for ONE reference polyline
    (agent.py:364-426 + utils/frenetix_handler.py:66-125; the C++ frenetix arithmetic is restated from
    the published Werling quartic/quintic scheme -- PARITY UNPINNED).  ``path`` is rounded to float32
    like the kernel input; vertices closer than ``MIN_CHORD`` to their predecessor are dropped, and a path left
    with fewer than 2 vertices gives sample -1 and zero rows (as the kernel).  Returns dict of [T] arrays and the
    selected sample index."""
    pts = np.asarray(path, dtype=np.float64).astype(np.float32).astype(np.float64).reshape(-1, 2)
    # a vertex closer than MIN_CHORD to its input predecessor is dropped (the heading of a zero chord is atan2(0, 0))
    dp = np.diff(pts, axis=0)
    pts = pts[np.concatenate(([True], ~(dp[:, 0] * dp[:, 0] + dp[:, 1] * dp[:, 1] < MIN_CHORD * MIN_CHORD)))[:len(pts)]]
    if len(pts) < 2:
        T = int(horizon / dt) + 1
        z = np.zeros(T)
        return {"x": z, "y": z.copy(), "yaw": z.copy(), "v": z.copy(), "var": z.copy(), "sample": -1, "s0": 0.0, "d0": 0.0}
    seg = np.diff(pts, axis=0)
    ln = np.hypot(seg[:, 0], seg[:, 1])
    cum = np.concatenate(([0.0], np.cumsum(ln)))
    n = len(pts)
    # projection
    best = (np.inf, 0.0, 0.0)
    for j in range(n - 1):
        if ln[j] <= 0:
            continue
        u = ((x0 - pts[j, 0]) * seg[j, 0] + (y0 - pts[j, 1]) * seg[j, 1]) / ln[j] ** 2
        uc = u if ((j == 0 and u < 0) or (j == n - 2 and u > 1)) else min(max(u, 0.0), 1.0)
        q = pts[j] + uc * seg[j]
        dist = np.hypot(x0 - q[0], y0 - q[1])
        if dist < best[0]:
            best = (dist, cum[j] + uc * ln[j], (seg[j, 0] * (y0 - pts[j, 1]) - seg[j, 1] * (x0 - pts[j, 0])) / ln[j])
    s0, d0 = best[1], best[2]
    T = int(horizon / dt) + 1
    t = np.arange(T) * dt
    head = np.arctan2(seg[:, 1], seg[:, 0])

    def frenet(sd1, d1):
        a3, a4 = (sd1 - v0) / t1 ** 2, (v0 - sd1) / (2 * t1 ** 3)
        tc = np.minimum(t, t1)
        s = s0 + v0 * tc + a3 * tc ** 3 + a4 * tc ** 4 + np.where(t > t1, sd1 * (t - t1), 0.0)
        sd = np.where(t < t1, v0 + 3 * a3 * tc ** 2 + 4 * a4 * tc ** 3, sd1)
        if v0 < 0.5:                     # low-velocity mode (frenetix_handler.py:91-95): lateral quintic over arc length
            s1 = s0 + v0 * t1 + a3 * t1 ** 3 + a4 * t1 ** 4
            span = max(s1 - s0, 1e-9)
            tau = np.clip((s - s0) / span, 0.0, 1.0)
            scale = sd / span
        else:
            tau = tc / t1
            scale = 1.0 / t1
        inside = (t < t1) | (v0 < 0.5)   # low-velocity mode: d follows the covered arc length at every t
        d = np.where(inside, d0 + (d1 - d0) * (10 * tau ** 3 - 15 * tau ** 4 + 6 * tau ** 5), d1)
        dd = np.where(inside, (d1 - d0) * scale * (30 * tau ** 2 - 60 * tau ** 3 + 30 * tau ** 4), 0.0)
        return s, sd, d, dd

    def lookup(s):
        j = np.clip(np.searchsorted(cum, s, side="right") - 1, 0, n - 2)
        kap = np.zeros_like(s)
        ok = j + 2 < n
        jj = np.where(ok, j, 0)
        dh = head[np.minimum(jj + 1, n - 2)] - head[jj]
        dh -= 2 * np.pi * np.rint(dh / (2 * np.pi))
        kap = np.where(ok, dh / (0.5 * (cum[np.minimum(jj + 2, n - 1)] - cum[jj])), 0.0)
        return j, kap

    best_k, best_var, keep = 0, np.inf, None
    for smp in range(9):
        sd1, d1 = v0 * (0.8 + 0.2 * (smp // 3)), -0.5 + 0.5 * (smp % 3)
        s, sd, d, dd = frenet(sd1, d1)
        j, kap = lookup(s)
        vl = sd * (1 - kap * d)
        v = np.sqrt(vl ** 2 + dd ** 2)
        var = max(np.mean(v * v) - np.mean(v) ** 2, 0.0)
        if var < best_var - 1e-15:
            best_k, best_var, keep = smp, var, (s, sd, d, dd, j, kap, vl, v)
    s, sd, d, dd, j, kap, vl, v = keep
    l = np.maximum(cum[j + 1] - cum[j], 1e-12)
    u = (s - cum[j]) / l
    tx, ty = seg[j, 0] / l, seg[j, 1] / l
    k = np.arange(T)
    return {"x": pts[j, 0] + u * seg[j, 0] - d * ty, "y": pts[j, 1] + u * seg[j, 1] + d * tx,
            "yaw": np.arctan2(ty, tx) + np.arctan2(dd, vl), "v": v, "var": var0 * np.power(var_factor, k),
            "sample": best_k, "s0": s0, "d0": d0}


# ------------------------------------------------------------------------------------------------
PT_IN_SENSOR, PT_ON_ROAD, PT_SHADOWED, PT_IN_OBSTACLE, PT_VISIBLE, PT_OCCLUDED, PT_FOCUS_SHADOW, PT_FOCUS_NEAR = \
    1, 2, 4, 8, 16, 32, 64, 128


def points_in_polygon(P, poly):
    """Even-odd rule in float64 for points [M,2] against one open ring [V,2]."""
    P = np.asarray(P, dtype=np.float64).reshape(-1, 2)
    poly = np.asarray(poly, dtype=np.float64).reshape(-1, 2)
    x, y = P[:, 0][:, None], P[:, 1][:, None]
    x1, y1 = poly[:, 0][None], poly[:, 1][None]
    x0, y0 = np.roll(poly[:, 0], 1)[None], np.roll(poly[:, 1], 1)[None]
    cond = (y0 > y) != (y1 > y)
    with np.errstate(divide="ignore", invalid="ignore"):
        xin = (x1 - x0) * (y - y0) / (y1 - y0) + x0
    return (np.sum(cond & (x < xin), axis=1) % 2).astype(bool)


def point_blockers(P, ego_xy, rect, flags, boundary, chunk=2048):
    """First opaque thing the segment ego -> P meets (float64): the owner (obstacle index or HIT_BOUNDARY) of the
    crossing with the smallest parameter along the segment (closed edges, first in edge order on ties), otherwise the
    lowest-index opaque obstacle that contains P (closed), otherwise HIT_NONE.  Returns (blocker [M], t12 [M, 2]): t12
    holds the segment parameters of the two nearest crossings (inf where there are fewer), so callers can tell
    near-ties apart."""
    P = np.asarray(P, dtype=np.float64).reshape(-1, 2) - np.asarray(ego_xy, dtype=np.float64)[:2]
    segs, owner = _edges(ego_xy, rect, flags, boundary)
    M = len(P)
    out = np.full(M, HIT_NONE, dtype=np.int64)
    t12 = np.full((M, 2), np.inf)
    if len(segs):
        ax, ay = segs[None, :, 0], segs[None, :, 1]
        ex, ey = segs[None, :, 2] - ax, segs[None, :, 3] - ay
        for c0 in range(0, M, chunk):
            px, py = P[c0:c0 + chunk, 0:1], P[c0:c0 + chunk, 1:2]
            D = px * ey - py * ex
            with np.errstate(divide="ignore", invalid="ignore"):
                t = (ax * ey - ay * ex) / D
                u = (ax * py - ay * px) / D
            t = np.where((D != 0) & (t >= 0) & (t <= 1) & (u >= 0) & (u <= 1), t, np.inf)
            j = t.argmin(1)
            hit = np.isfinite(t[np.arange(len(t)), j])
            out[c0:c0 + chunk] = np.where(hit, owner[j], HIT_NONE)
            t12[c0:c0 + chunk] = np.sort(t, 1)[:, :2] if t.shape[1] > 1 else np.concatenate((t, np.full_like(t, np.inf)), 1)
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    flags = np.asarray(flags).reshape(-1)
    container = np.full(M, HIT_NONE, dtype=np.int64)
    for o in range(len(rect) - 1, -1, -1):              # descending: the lowest index is written last
        if not (flags[o] & RECT_EXISTS) or (flags[o] & RECT_TRANSPARENT):
            continue
        cs, sn = np.cos(rect[o, 2]), np.sin(rect[o, 2])
        dx, dy = P[:, 0] - (rect[o, 0] - ego_xy[0]), P[:, 1] - (rect[o, 1] - ego_xy[1])
        inside = (np.abs(dx * cs + dy * sn) <= rect[o, 3]) & (np.abs(-dx * sn + dy * cs) <= rect[o, 4])
        container = np.where(inside, o, container)
    return np.where(out == HIT_NONE, container, out), t12


def classify_points(P, ego, rect, flags, boundary, polygons, sensor_radius, fov_deg, occluded_radius, focus=-1,
                    focus_margin=0.0):
    """Point-wise evaluation of the reference's visible / occluded area construction (float64):
    visible_area = road ∩ sector − border-edge shadow quads − obstacles − obstacle shadows
    (sensor_model.py:103-193), occluded_area = (±90° sector of radius 1.5 R) ∩ road − visible_area
    (sensor_model.py:85-93), obstacle_occlusions[id] = shadow(id) − obstacle(id) (sensor_model.py:182-183).
    Returns (flags uint32 [M], lanelet bit mask uint64 [M])."""
    P = np.asarray(P, dtype=np.float64).reshape(-1, 2)
    ego = np.asarray(ego, dtype=np.float64)
    e = ego[:2]
    d = P - e
    r = np.hypot(d[:, 0], d[:, 1])
    rel = (np.arctan2(d[:, 1], d[:, 0]) - ego[2] + np.pi) % (2 * np.pi) - np.pi
    in_sensor = r <= sensor_radius
    if fov_deg < 359.9:
        in_sensor &= np.abs(rel) <= np.radians(fov_deg) / 2
    shadow = np.zeros(len(P), dtype=bool)
    if boundary is not None:
        for b in np.asarray(boundary, dtype=np.float64).reshape(-1, 4):
            v1, v2 = b[:2], b[2:]
            if np.allclose(v1, v2):
                continue
            shadow |= _in_convex_quad(P, [v1, v2, v2 + 100 * (v2 - e), v1 + 100 * (v1 - e)])
    rect = np.asarray(rect, dtype=np.float64).reshape(-1, 5)
    flags = np.asarray(flags).reshape(-1)
    cor = rect_corners(rect)
    in_obst = np.zeros(len(P), dtype=bool)
    focus_shadow = np.zeros(len(P), dtype=bool)
    focus_near = np.zeros(len(P), dtype=bool)
    for o in range(len(rect)):
        if not (flags[o] & RECT_EXISTS) or (flags[o] & RECT_TRANSPARENT):
            continue
        c1, c2 = identify_projection_points(e, cor[o])
        u1 = (c1 - e) / np.linalg.norm(c1 - e)
        u2 = (c2 - e) / np.linalg.norm(c2 - e)
        wedge = _in_convex_quad(P, [c1, c2, c2 + u2 * 100, c1 + u1 * 100])
        inside = _in_convex_quad(P, cor[o])
        shadow |= wedge & ~inside
        in_obst |= inside
        if o == focus:
            focus_shadow = wedge & ~inside
            # distance to the rectangle (0 inside) <= margin  ==  within polygon.buffer(margin) (round joins)
            cs, sn = np.cos(rect[o, 2]), np.sin(rect[o, 2])
            dl = P - rect[o, :2]
            lx, ly = dl[:, 0] * cs + dl[:, 1] * sn, -dl[:, 0] * sn + dl[:, 1] * cs
            focus_near = np.hypot(np.maximum(np.abs(lx) - rect[o, 3], 0), np.maximum(np.abs(ly) - rect[o, 4], 0)) <= focus_margin
    lan = np.zeros(len(P), dtype=np.uint64)
    on_road = np.zeros(len(P), dtype=bool)
    for i, poly in enumerate(polygons):
        m = points_in_polygon(P, poly)
        on_road |= m
        if i < 64:
            lan |= np.where(m, np.uint64(1) << np.uint64(i), np.uint64(0))
    visible = in_sensor & on_road & ~shadow & ~in_obst
    occluded = on_road & ~visible & (np.abs(rel) <= np.pi / 2) & (r <= occluded_radius)
    f = (in_sensor * PT_IN_SENSOR + on_road * PT_ON_ROAD + shadow * PT_SHADOWED + in_obst * PT_IN_OBSTACLE
         + visible * PT_VISIBLE + occluded * PT_OCCLUDED + focus_shadow * PT_FOCUS_SHADOW
         + focus_near * PT_FOCUS_NEAR).astype(np.uint32)
    return f, lan
