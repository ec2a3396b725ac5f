"""Helpers of the ray-cast tests: run ``raycast_frames`` on host inputs, certify its frames with
``VO.certify_raycast`` and compare two casts of the same frames.

Two casts of one frame agree bit for bit except at exact ties: the update ``t.x < bq * D`` is not exactly a minimum of
quotients, and a CTA stages a frame's edges in an order that depends on its warps' atomics, so at a corner where two
edges meet a ray at the same float32 range either edge (and either owner) may be reported, and the ranges may differ in
the last bits.  ``assert_same_or_tied`` accepts such a ray only when both answers pass the certificate and their ranges
lie within 2 float32 ulp."""
import numpy as np

from oracle import visibility_oracle as VO


def f32(a):
    """Round to float32 and back: the kernel and the float64 certificate then see the same numbers."""
    return None if a is None else np.asarray(a, dtype=np.float64).astype(np.float32).astype(np.float64)


def cast(ego, rect, flags, boundary, R, fov, n_rays, stats=None):
    """ego [F,3], rect [F,O,5], flags [F,O] host arrays -> host (range [F,N], hit [F,N], visible [F,O])."""
    import torch
    from frenetix_occlusion_b200.visibility import raycast_frames
    res = raycast_frames(ego, rect, flags, boundary, R, fov, n_rays, stats=stats)
    torch.cuda.synchronize()
    return res.range.cpu().numpy(), res.hit.cpu().numpy(), res.visible.cpu().numpy()


def certify(out, f, ego, rect, flags, boundary, R, fov, n_rays, what=""):
    """Frame f of cast output ``out`` passes the certificate (ego [3], rect [O,5], flags [O] of that frame)."""
    cert = VO.certify_raycast(out[0][f], out[1][f], out[2][f], ego, rect, flags, boundary, R, fov, n_rays)
    assert cert["n_fail"] == 0, f"{what} frame {f}: " + VO.certificate_failures(cert)


def assert_same_or_tied(x, y, frame, R, fov, n_rays, what="", ulp=2):
    """x, y: (range, hit, visible) of the same frames.  ``frame(f)`` -> (ego, rect, flags, boundary) of frame f.
    Bit-identical, except rays whose two answers both pass the certificate and lie within ``ulp`` float32 ulp (None:
    any distance -- for inputs that describe the same geometry with different float32 numbers), and visible flags of
    frames whose differing answers both pass the certificate."""
    rx, ry = x[0].view(np.int32).astype(np.int64), y[0].view(np.int32).astype(np.int64)
    bad = (rx != ry) | (x[1] != y[1])
    if ulp is not None:
        far = np.abs(rx - ry) > ulp
        assert not far.any(), f"{what}: ranges differ by more than {ulp} ulp at {np.argwhere(far)[:5].tolist()}"
    vbad = np.flatnonzero((x[2] != y[2]).any(1))
    for f in np.flatnonzero(bad.any(1)):
        ego, rect, flags, bnd = frame(f)
        rays = np.flatnonzero(bad[f])
        for o in (x, y):
            cert = VO.certify_raycast(o[0][f, rays], o[1][f, rays], None, ego, rect, flags, bnd, R, fov, n_rays, rays=rays)
            assert cert["n_fail"] == 0, f"{what} frame {f}, differing rays {rays[:8]}: " + VO.certificate_failures(cert)
    for f in vbad:
        ego, rect, flags, bnd = frame(f)
        for o in (x, y):
            certify(o, f, ego, rect, flags, bnd, R, fov, n_rays, what=what + " (visible flags differ)")
