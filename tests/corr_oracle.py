"""Float64 oracle of the dense metric core for predictions with full 2x2 covariances (test infrastructure).

A case's agents may carry ``cov`` [T_a, 2, 2] (the prediction's ``cov_list``) in addition to the fields of the case
format of ``oracle/ref_runner.py``.  The collision probability then follows the reference's
``mvnun(lower, upper, mean, cov[i-1])`` (collision_probability.py:94-122) with the full covariance: each of the nine
ego-box x obstacle-point terms is the mass of N(mu, Sigma) over the box, / 3; an all-zero matrix is 0.1 I
(collision_probability.py:85-87).  Everything else -- the 5 m gate, the index offsets, DCE, TTC, harm, BE, the
thresholds -- is ``oracle.metric_oracle`` unchanged: ``evaluate_bundle`` runs it with this module's
``collision_probability`` in place of the diagonal one.

The rectangle masses come from a vectorised float64 port of Genz's BVNU (``bvn_rect``); ``test_metric_corr`` pins it to
``oracle.ref_shims.mvnun`` (scipy's ``multivariate_normal.cdf``, the stand-in oracle A uses for the reference's
``mvnun``) and to a 1-D quadrature of the conditional form.
"""
from unittest import mock

import numpy as np
from numpy.polynomial.legendre import leggauss
from scipy.special import ndtr

from oracle import metric_oracle as MO

_GL = {n: leggauss(n) for n in (6, 12, 20)}   # Gauss-Legendre rules of BVNU, by |r| < 0.3 / < 0.75 / else


def bvn_upper(h, k, r):
    """P(X > h, Y > k) of a standard bivariate normal with correlation r (arrays, |r| < 1; NaN otherwise)."""
    h, k, r = (np.array(v, dtype=np.float64) for v in np.broadcast_arrays(h, k, r))
    out = np.full(h.shape, np.nan)
    ar = np.abs(r)
    with np.errstate(all="ignore"):
        for n, sel in ((6, ar < 0.3), (12, (ar >= 0.3) & (ar < 0.75)), (20, ar >= 0.75)):
            x, w = _GL[n]
            lo = sel & (ar < 0.925)
            if lo.any():                               # Drezner-Wesolowsky: integral over asin(r)
                hh, kk, rr = h[lo], k[lo], r[lo]
                hk, hs, asr = hh * kk, 0.5 * (hh * hh + kk * kk), np.arcsin(rr)
                sn = np.sin(0.5 * asr[:, None] * (x[None] + 1.0))
                s = (w[None] * np.exp((sn * hk[:, None] - hs[:, None]) / (1.0 - sn * sn))).sum(1)
                out[lo] = s * asr / (4.0 * np.pi) + ndtr(-hh) * ndtr(-kk)
            hi = sel & (ar >= 0.925) & (ar < 1.0)
            if hi.any():                               # expansion around |r| = 1
                hh, rr = h[hi], r[hi]
                kk = np.where(rr < 0, -k[hi], k[hi])
                hk = hh * kk
                as_ = (1.0 - rr) * (1.0 + rr)
                a = np.sqrt(as_)
                bs = (hh - kk) ** 2
                c, d = (4.0 - hk) / 8.0, (12.0 - hk) / 16.0
                bvn = a * np.exp(-0.5 * (bs / as_ + hk)) * (1 - c * (bs - as_) * (1 - d * bs / 5) / 3 + c * d * as_ * as_ / 5)
                b = np.sqrt(bs)
                tail = np.exp(-0.5 * hk) * np.sqrt(2 * np.pi) * ndtr(-b / a) * b * (1 - c * bs * (1 - d * bs / 5) / 3)
                bvn = np.where(hk > -160.0, bvn - tail, bvn)
                a2 = 0.5 * a[:, None]
                xs = (a2 * (x[None] + 1.0)) ** 2
                rs = np.sqrt(1.0 - xs)
                t = a2 * w[None] * (np.exp(-bs[:, None] / (2 * xs) - hk[:, None] / (1 + rs)) / rs
                                    - np.exp(-0.5 * (bs[:, None] / xs + hk[:, None])) * (1 + c[:, None] * xs * (1 + d[:, None] * xs)))
                bvn = -(bvn + t.sum(1)) / (2 * np.pi)
                neg = -bvn + np.where(kk > hh, np.where(hh < 0, ndtr(kk) - ndtr(hh), ndtr(-hh) - ndtr(-kk)), 0.0)
                out[hi] = np.where(rr > 0, bvn + ndtr(-np.maximum(hh, kk)), neg)
    return out


def bvn_rect(a1, b1, a2, b2, r):
    """Mass of a standard bivariate normal with correlation r over [a1, b1] x [a2, b2], combined on the tails (a
    coordinate whose interval lies mostly below the mean is reflected and r changes sign)."""
    a1, b1, a2, b2, r = (np.array(v, dtype=np.float64) for v in np.broadcast_arrays(a1, b1, a2, b2, r))
    f = a1 + b1 < 0
    a1, b1, r = np.where(f, -b1, a1), np.where(f, -a1, b1), np.where(f, -r, r)
    f = a2 + b2 < 0
    a2, b2, r = np.where(f, -b2, a2), np.where(f, -a2, b2), np.where(f, -r, r)
    return bvn_upper(a1, a2, r) - bvn_upper(b1, a2, r) - bvn_upper(a1, b2, r) + bvn_upper(b1, b2, r)


def _covariances(case, A, Tm):
    """[A, Tm, 3] (var_x, var_y, cov_xy) of every state; an agent without ``cov`` has var * I."""
    out = np.zeros((A, Tm, 3))
    out[..., :2] = 0.1
    for k, a in enumerate(case["agents"]):
        n = len(np.asarray(a["yaw"]))
        if "cov" in a:
            c = np.asarray(a["cov"], dtype=np.float64)
            out[k, :n] = np.stack((c[:, 0, 0], c[:, 1, 1], c[:, 0, 1]), -1)
        else:
            out[k, :n, 0] = out[k, :n, 1] = a["var"]
    return out


def collision_probability(case):
    """``oracle.metric_oracle.collision_probability`` with the full covariance of state i-1."""
    ego = np.asarray(case["ego"], dtype=np.float64)
    N, T, _ = ego.shape
    A, Ta, Tm, pos, yaw, vel, var = MO._stack_agents(case)
    cov = _covariances(case, A, Tm)
    L, W = case["vehicle"]["length"], case["vehicle"]["width"]
    cp = np.zeros((N, A, max(T - 1, 0)))
    inside = np.zeros((N, A, max(T - 1, 0)), dtype=bool)
    gate_margin = np.full((N, A, max(T - 1, 0)), np.inf)
    for a in range(A):
        nmax = min(T, Ta[a])
        if nmax < 2:
            continue
        i = np.arange(1, nmax)
        lb = case["agents"][a]["buf_length"]
        p = pos[a, i - 1]
        h = np.stack((np.cos(yaw[a, i]), np.sin(yaw[a, i])), -1) * lb / 2
        mus = np.stack((p, p + h, p - h), 0)                          # [3, n, 2]
        e = ego[:, i, 0:2]
        d = np.sqrt(((mus[None] - e[:, None]) ** 2).sum(-1))
        gate = d.min(1) > 5.0
        vx, vy, cxy = cov[a, i - 1].T.copy()
        zero = (vx == 0) & (vy == 0) & (cxy == 0)
        vx[zero], vy[zero] = 0.1, 0.1                                 # :85-87
        sx, sy = np.sqrt(vx), np.sqrt(vy)
        with np.errstate(divide="ignore", invalid="ignore"):
            rho = cxy / (sx * sy)
        th = ego[:, i, 2]
        off = np.stack((np.cos(th), np.sin(th)), -1) * (L / 3.0)
        cen = np.stack((e, e + off, e - off), 1)                      # [N, 3, n, 2]
        half = np.array([L / 6.0, W / 2.0])
        lo = (cen - half)[:, None] - mus[None, :, None]               # [N, mu(3), box(3), n, 2]
        hi = (cen + half)[:, None] - mus[None, :, None]
        nn, jj = np.nonzero(~gate)                                    # the nine masses of the gated steps only
        lo, hi = lo[nn, :, :, jj], hi[nn, :, :, jj]                   # [M, 3, 3, 2]
        s_x, s_y, r = sx[jj, None, None], sy[jj, None, None], rho[jj, None, None]
        prob = np.zeros(gate.shape)
        prob[nn, jj] = bvn_rect(lo[..., 0] / s_x, hi[..., 0] / s_x, lo[..., 1] / s_y, hi[..., 1] / s_y, r).sum((1, 2)) / 3.0
        cp[:, a, i - 1] = prob
        inside[:, a, i - 1] = ~gate
        gate_margin[:, a, i - 1] = np.abs(d.min(1) - 5.0)
    return cp, inside, gate_margin


def evaluate_bundle(case, want_detail: bool = True):
    """``oracle.metric_oracle.evaluate_bundle`` with the full-covariance collision probability."""
    with mock.patch.object(MO, "collision_probability", collision_probability):
        return MO.evaluate_bundle(case, want_detail)


def add_correlations(case, seed, extremes=(-0.99, 0.99)):
    """Give every agent of ``case`` correlated covariances: per state var_x != var_y around its diagonal variance and
    rho ~ U(-0.99, 0.99), with ``extremes`` placed on the first agents' states.  Values are float32-representable (the
    kernels read float32).  Returns the case."""
    rng = np.random.default_rng(seed)
    for k, a in enumerate(case["agents"]):
        v = np.asarray(a["var"], dtype=np.float64)
        n = len(v)
        vx = v * rng.uniform(0.3, 3.0, n)
        vy = v * rng.uniform(0.3, 3.0, n)
        rho = rng.uniform(-0.99, 0.99, n)
        if k < len(extremes):
            rho[::2] = extremes[k]
        f = lambda z: z.astype(np.float32).astype(np.float64)      # noqa: E731
        vx, vy = f(vx), f(vy)
        c = f(rho * np.sqrt(vx * vy))
        a["cov"] = np.stack((np.stack((vx, c), -1), np.stack((c, vy), -1)), -2)
    return case
