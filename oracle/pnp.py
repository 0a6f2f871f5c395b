"""RANSAC P3P over a 2D-3D match list (csrc/pnp.cu) restated in NumPy — TEST INFRASTRUCTURE ONLY.

The sampler (oracle/fundamental.py's, with 4 rows), the Lambda Twist P3P solve, the choice by the 4th row
and the fp32 inlier test follow the kernel operation by operation: NumPy's element-wise loops round every
product, sum, quotient and square root separately (no contraction), as the kernel's __dmul_rn / __dadd_rn /
__ddiv_rn / __dsqrt_rn and __fmul_rn / __fadd_rn / __frcp_rn do, and the bisection, the Gauss-Newton steps
and the solution order are the kernel's.  Hypotheses, per-sample inlier counts, the best sample and its
inlier mask are therefore bit-identical to the device's.  The Levenberg-Marquardt refinement is restated
in float64 with NumPy sums (the kernel: fixed-order block reductions, CUDA's sin / cos), so the refined
pose agrees to rounding.

A row is (X, Y, Z, u, v): the 3-D point and the keypoint it is matched to, float32.
"""

import math

import numpy as np

from .fundamental import sample_rows
from .geometry import t2_of

CUBIC_BISECT = 100
GN_STEPS = 5
COLLINEAR_TOL = 1e-12
MIN_REFINE_ROWS = 4
NP = 6


def _dot3(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1],
                     a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], -1)


def _root2(b, c):
    """Roots of x^2 + b x + c, the discriminant clamped at 0, in Lambda Twist's order."""
    v = b * b - 4.0 * c
    y = np.sqrt(np.where(v > 0.0, v, 0.0))
    sp, sm = -b + y, -b - y
    r1 = np.where(b < 0.0, 0.5 * sp, (2.0 * c) / sm)
    r2 = np.where(b < 0.0, (2.0 * c) / sp, 0.5 * sm)
    return r1, r2


def _eigvec(A, e, mx0011, x01sq, prec0, prec1):
    den = ((e * (A[0] + A[3]) + mx0011) - e * e) + x01sq
    tmp = 1.0 / den
    a1 = (-(e * A[2] + prec0)) * tmp
    a2 = (-(e * A[4] + prec1)) * tmp
    rn = 1.0 / np.sqrt((a1 * a1 + a2 * a2) + 1.0)
    return np.stack([a1 * rn, a2 * rn, rn], -1)


def _gn_cost(l, a12, a13, a23, b12, b13, b23):
    r0 = ((l[..., 0] * l[..., 0] + l[..., 1] * l[..., 1]) + (b12 * l[..., 0]) * l[..., 1]) - a12
    r1 = ((l[..., 0] * l[..., 0] + l[..., 2] * l[..., 2]) + (b13 * l[..., 0]) * l[..., 2]) - a13
    r2 = ((l[..., 1] * l[..., 1] + l[..., 2] * l[..., 2]) + (b23 * l[..., 1]) * l[..., 2]) - a23
    return (np.abs(r0) + np.abs(r1)) + np.abs(r2), (r0, r1, r2)


def _refine_depths(l, a12, a13, a23, b12, b13, b23):
    act = np.ones(l.shape[:-1], bool)
    for _ in range(GN_STEPS):
        c0, (r0, r1, r2) = _gn_cost(l, a12, a13, a23, b12, b13, b23)
        act &= ~(c0 < 1e-10)
        l0, l1, l2 = l[..., 0], l[..., 1], l[..., 2]
        v0, v1 = 2.0 * l0 + b12 * l1, 2.0 * l1 + b12 * l0
        v3, v5 = 2.0 * l0 + b13 * l2, 2.0 * l2 + b13 * l0
        v7, v8 = 2.0 * l1 + b23 * l2, 2.0 * l2 + b23 * l1
        det = 1.0 / (((-v0) * v5) * v7 - (v1 * v3) * v8)
        j0 = (((-v5) * v7) * r0 + ((-v1) * v8) * r1) + (v1 * v5) * r2
        j1 = (((-v3) * v8) * r0 + (v0 * v8) * r1) + ((-v0) * v5) * r2
        j2 = ((v3 * v7) * r0 + ((-v0) * v7) * r1) + ((-v1) * v3) * r2
        ln = np.stack([l0 - det * j0, l1 - det * j1, l2 - det * j2], -1)
        cn, _ = _gn_cost(ln, a12, a13, a23, b12, b13, b23)
        act &= ~(cn > c0)
        l = np.where(act[..., None], ln, l)
    return l


def p3p(y, x):
    """Lambda Twist on S samples: bearings y (S,3,3) unit, points x (S,3,3) -> Rs (S,4,9), ts (S,4,3),
    valid (S,4) in the kernel's solution order (sign +v then -v, each with tau1 then tau2)."""
    S = y.shape[0]
    with np.errstate(all="ignore"):
        b12, b13, b23 = -2.0 * _dot3(y[:, 0], y[:, 1]), -2.0 * _dot3(y[:, 0], y[:, 2]), -2.0 * _dot3(y[:, 1], y[:, 2])
        d12, d13, d23 = x[:, 0] - x[:, 1], x[:, 0] - x[:, 2], x[:, 1] - x[:, 2]
        c = _cross(d12, d13)
        a12, a13, a23 = _dot3(d12, d12), _dot3(d13, d13), _dot3(d23, d23)
        cc = _dot3(c, c)
        ok = cc > (COLLINEAR_TOL * a12) * a13
        c31, c23, c12 = -0.5 * b13, -0.5 * b23, -0.5 * b12
        blob = (c12 * c23) * c31 - 1.0
        s31, s23, s12 = 1.0 - c31 * c31, 1.0 - c23 * c23, 1.0 - c12 * c12
        p3 = a13 * (a23 * s31 - a13 * s23)
        p2 = ((((2.0 * blob) * a23) * a13 + (a13 * (2.0 * a12 + a13)) * s23) + (a23 * (a23 - a12)) * s31)
        p1 = (((a23 * (a13 - a23)) * s12 - (a12 * a12) * s23) - (2.0 * a12) * (blob * a23 + a13 * s23))
        p0 = a12 * (a12 * s23 - a23 * s12)
        ok &= (p3 != 0.0) & np.isfinite(p3)
        k2, k1, k0 = p2 / p3, p1 / p3, p0 / p3
        B = 1.0 + np.fmax(np.fmax(np.abs(k2), np.abs(k1)), np.abs(k0))
        ok &= np.isfinite(B)
        lo, hi = -B, B.copy()
        for _ in range(CUBIC_BISECT):
            m = (lo + hi) * 0.5
            f = (((m + k2) * m + k1) * m) + k0
            neg = f < 0.0
            lo, hi = np.where(neg, m, lo), np.where(neg, hi, m)
        g = (lo + hi) * 0.5
        A = [a23 * (1.0 - g), (a23 * b12) * 0.5, ((a23 * b13) * g) * -0.5, (a23 - a12) + a13 * g,
             (b23 * (a13 * g - a12)) * 0.5, g * (a13 - a23) - a12]
        x01sq = A[1] * A[1]
        eb = ((-A[0]) - A[3]) - A[5]
        ec = ((((-x01sq) - A[2] * A[2]) - A[4] * A[4]) + A[0] * (A[3] + A[5])) + A[3] * A[5]
        e1, e2 = _root2(eb, ec)
        sw = np.abs(e1) < np.abs(e2)
        e1, e2 = np.where(sw, e2, e1), np.where(sw, e1, e2)
        mx0011 = (-A[0]) * A[3]
        prec0 = A[1] * A[4] - A[2] * A[3]
        prec1 = A[1] * A[2] - A[0] * A[4]
        v1 = _eigvec(A, e1, mx0011, x01sq, prec0, prec1)
        v2 = _eigvec(A, e2, mx0011, x01sq, prec0, prec1)
        q = -(e2 / e1)
        sv = np.sqrt(np.where(q > 0.0, q, 0.0))
        Ls = np.zeros((S, 4, 3))
        valid = np.zeros((S, 4), bool)
        for sgn in range(2):
            s = sv if sgn == 0 else -sv
            w2 = 1.0 / (s * v2[:, 0] - v1[:, 0])
            w0 = (v1[:, 1] - s * v2[:, 1]) * w2
            w1 = (v1[:, 2] - s * v2[:, 2]) * w2
            a = 1.0 / ((((a13 - a12) * w1) * w1 - (a12 * b13) * w1) - a12)
            bb = ((((a13 * b12) * w1 - (a12 * b13) * w0) - ((2.0 * w0) * w1) * (a12 - a13)) * a)
            cq = ((((a13 - a12) * w0) * w0 + (a13 * b12) * w0) + a13) * a
            real = (bb * bb - 4.0 * cq) >= 0.0
            taus = _root2(bb, cq)
            for k in range(2):
                tau = taus[k]
                d = a23 / (tau * (b23 + tau) + 1.0)
                l2 = np.sqrt(d)
                l3 = tau * l2
                l1 = w0 * l2 + w1 * l3
                v = ok & real & (tau > 0.0) & (d > 0.0) & (l1 >= 0.0)
                slot = 2 * sgn + k
                Ls[:, slot] = np.stack([l1, l2, l3], -1)
                valid[:, slot] = v
        Ls = np.where(valid[..., None], Ls, 1.0)
        bc = [v[:, None] for v in (a12, a13, a23, b12, b13, b23)]
        Ls = _refine_depths(Ls, *bc)
        Xi = np.stack([_cross(d13, c) / cc[:, None], _cross(c, d12) / cc[:, None], c / cc[:, None]], 1)   # (S,3,3)
        ry = y[:, None, :, :] * Ls[..., :, None]                  # (S,4,3,3): ry[s, i, k] = y_k l_k
        yd1, yd2 = ry[:, :, 0] - ry[:, :, 1], ry[:, :, 0] - ry[:, :, 2]
        yc = _cross(yd1, yd2)
        Rs = np.empty((S, 4, 9))
        for r in range(3):
            for j in range(3):
                Rs[:, :, 3 * r + j] = ((yd1[..., r] * Xi[:, None, 0, j] + yd2[..., r] * Xi[:, None, 1, j]) +
                                       yc[..., r] * Xi[:, None, 2, j])
        ts = np.empty((S, 4, 3))
        for r in range(3):
            ts[:, :, r] = ry[:, :, 0, r] - _dot3(Rs[:, :, 3 * r:3 * r + 3], x[:, None, 0])
    return Rs, ts, valid


def bearings(uv, camera):
    """(..., 2) pixels -> (..., 3) unit bearings, in the kernel's order."""
    fx, fy, cx, cy = camera
    f0, f1 = (uv[..., 0] - cx) / fx, (uv[..., 1] - cy) / fy
    n = np.sqrt((f0 * f0 + f1 * f1) + 1.0)
    return np.stack([f0 / n, f1 / n, 1.0 / n], -1)


def sample_poses(rows, camera, samples, seed):
    """Poses of ``samples`` for a list of rows (n,5) float32 -> R (S,9), t (S,3) float64, ok (S,)."""
    rows = np.asarray(rows, dtype=np.float32).reshape(-1, 5)
    n = rows.shape[0]
    samples = np.asarray(samples)
    S = samples.shape[0]
    R, t, ok = np.zeros((S, 9)), np.zeros((S, 3)), np.zeros(S, bool)
    if n < 4 or S == 0:
        return R, t, ok
    idx, drawn = sample_rows(seed, n, samples, R=4)
    q = rows[np.where(drawn[:, None], idx, 0)].astype(np.float64)          # (S,4,5)
    fin = drawn & np.isfinite(q).all((1, 2))
    q = np.where(fin[:, None, None], q, 1.0)
    X, uv = q[..., :3], q[..., 3:]
    fx, fy, cx, cy = camera
    with np.errstate(all="ignore"):
        y = bearings(uv[:, :3], camera)
        Rs, ts, valid = p3p(y, X[:, :3])
        good = valid & np.isfinite(Rs).all(-1) & np.isfinite(ts).all(-1)
        for k in range(4):
            good &= (_dot3(Rs[..., 6:9], X[:, None, k]) + ts[..., 2]) > 0.0
        xc = _dot3(Rs[..., 0:3], X[:, None, 3]) + ts[..., 0]
        yc = _dot3(Rs[..., 3:6], X[:, None, 3]) + ts[..., 1]
        zc = _dot3(Rs[..., 6:9], X[:, None, 3]) + ts[..., 2]
        du = (fx * (xc / zc) + cx) - uv[:, None, 3, 0]
        dv = (fy * (yc / zc) + cy) - uv[:, None, 3, 1]
        e = du * du + dv * dv
    best = np.full(S, -1)
    be = np.zeros(S)
    for i in range(4):                                   # first strict minimum among the good solutions
        take = good[:, i] & ((best < 0) | (e[:, i] < be))
        best = np.where(take, i, best)
        be = np.where(take, e[:, i], be)
    ok = fin & (best >= 0)
    sel = np.where(ok, best, 0)
    R = np.where(ok[:, None], Rs[np.arange(S), sel], 0.0)
    t = np.where(ok[:, None], ts[np.arange(S), sel], 0.0)
    return R, t, ok


def sq_errors(h32, rows, camera):
    """Squared reprojection errors in the kernel's fp32 order: h32 (H,12) float32 (R row-major, t), rows
    (n,5) float32 -> (err (H,n), Zc (H,n)) float32."""
    fx, fy, cx, cy = (np.float32(v) for v in camera)
    h = [h32[:, k:k + 1] for k in range(12)]
    X, Y, Z, u, v = (rows[None, :, c] for c in range(5))
    xc = ((h[0] * X + h[1] * Y) + h[2] * Z) + h[9]
    yc = ((h[3] * X + h[4] * Y) + h[5] * Z) + h[10]
    zc = ((h[6] * X + h[7] * Y) + h[8] * Z) + h[11]
    iz = np.float32(1.0) / zc
    du = ((fx * xc) * iz + cx) - u
    dv = ((fy * yc) * iz + cy) - v
    return du * du + dv * dv, zc


def to32(R, t):
    return np.concatenate([np.asarray(R, np.float64).reshape(-1, 9), np.asarray(t, np.float64).reshape(-1, 3)],
                          1).astype(np.float32)


def inliers(R, t, rows, camera, threshold):
    """Inlier mask (n,) of one double pose after rounding it to fp32, as the kernel scores."""
    with np.errstate(all="ignore"):
        e, z = sq_errors(to32(R, t), np.asarray(rows, np.float32).reshape(-1, 5), camera)
        return (z[0] > 0) & (e[0] < t2_of(threshold))


def near_threshold(R, t, rows, camera, threshold, rel=1e-6):
    """Rows whose inlier decision under (R, t) sits within ``rel`` of the threshold or of Zc = 0."""
    with np.errstate(all="ignore"):
        e, z = sq_errors(to32(R, t), np.asarray(rows, np.float32).reshape(-1, 5), camera)
        t2 = float(t2_of(threshold))
        return (np.abs(e[0].astype(np.float64) - t2) <= rel * t2) | (np.abs(z[0]) <= rel * np.maximum(1.0, np.abs(t[2])))


# ---------------------------------------------------------------------------- refinement (float64)
def skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def exp_so3(w):
    th = math.sqrt(float(np.dot(w, w)))
    if not th > 0.0:
        return np.eye(3)
    K = skew(np.asarray(w) / th)
    return (np.eye(3) + math.sin(th) * K) + (1.0 - math.cos(th)) * (K @ K)


def residuals(R, t, rows, camera):
    """Reprojection residuals (2n,) in px: u rows then v rows."""
    fx, fy, cx, cy = camera
    q = np.asarray(rows, np.float64).reshape(-1, 5)
    Xc = q[:, :3] @ np.asarray(R).reshape(3, 3).T + t
    return np.concatenate([fx * (Xc[:, 0] / Xc[:, 2]) + cx - q[:, 3], fy * (Xc[:, 1] / Xc[:, 2]) + cy - q[:, 4]])


def jacobian(R, t, rows, camera):
    """d residuals / d(w, d) for R <- Exp(w) R, t <- t + d -> (2n, 6)."""
    fx, fy = camera[0], camera[1]
    q = np.asarray(rows, np.float64).reshape(-1, 5)
    rx = q[:, :3] @ np.asarray(R).reshape(3, 3).T
    Xc = rx + t
    iz = 1.0 / Xc[:, 2]
    z = np.zeros_like(iz)
    gu = np.stack([fx * iz, z, -(fx * Xc[:, 0] * iz) * iz], 1)
    gv = np.stack([z, fy * iz, -(fy * Xc[:, 1] * iz) * iz], 1)
    cols = [np.stack([z, -rx[:, 2], rx[:, 1]], 1), np.stack([rx[:, 2], z, -rx[:, 0]], 1),
            np.stack([-rx[:, 1], rx[:, 0], z], 1)]
    Ju = np.stack([(gu * c).sum(1) for c in cols], 1)
    Jv = np.stack([(gv * c).sum(1) for c in cols], 1)
    return np.concatenate([np.concatenate([Ju, gu], 1), np.concatenate([Jv, gv], 1)])


def refine(R, t, rows, camera, iters):
    """The kernel's LM trials over rows -> (R, t, cost before, cost after, accepted steps)."""
    R, t = np.asarray(R, np.float64).reshape(3, 3), np.asarray(t, np.float64).reshape(3)
    r = residuals(R, t, rows, camera)
    cost0 = cost = float(r @ r)
    accepted = 0
    if iters <= 0 or len(rows) < MIN_REFINE_ROWS:
        return R, t, cost0, cost, accepted
    J = jacobian(R, t, rows, camera)
    JtJ, Jtr = J.T @ J, J.T @ r
    lam = 1e-3 * (float(np.trace(JtJ)) / NP)
    for it in range(iters):
        A = JtJ + lam * np.diag(np.diag(JtJ))
        try:
            L = np.linalg.cholesky(A)
            x = -np.linalg.solve(L.T, np.linalg.solve(L, Jtr))
        except np.linalg.LinAlgError:
            x = None
        accept = False
        if x is not None and np.isfinite(x).all():
            Rn, tn = exp_so3(x[:3]) @ R, t + x[3:]
            with np.errstate(all="ignore"):
                rn = residuals(Rn, tn, rows, camera)
            c = float(rn @ rn)
            accept = c < cost
        if accept:
            R, t, cost, lam = Rn, tn, c, lam / 10.0
            accepted += 1
            if it + 1 < iters:
                r = residuals(R, t, rows, camera)
                J = jacobian(R, t, rows, camera)
                JtJ, Jtr = J.T @ J, J.T @ r
        else:
            lam = lam * 10.0
    return R, t, cost0, cost, accepted


def ransac_pnp(rows, camera, iters=1024, threshold=3.0, seed=0, refine_iters=10):
    """One list of rows (n,5) float32 (X, Y, Z, u, v in list order; NaN where a row is not usable), camera
    (fx, fy, cx, cy) -> dict: hyp_count (iters,) (-1 degenerate), best (-1 none), hyp_mask (n,) before the
    refinement, refit_used, R (3,3), t (3,) (zeros: no model, also when the best sample has no inlier),
    rms (2,), mask (n,) final inliers, band (n,) rows within 1e-6 of the threshold under the final pose."""
    rows = np.ascontiguousarray(np.asarray(rows, dtype=np.float32).reshape(-1, 5))
    n = rows.shape[0]
    Rh, th, ok = sample_poses(rows, camera, np.arange(iters), seed)
    count = np.full(iters, -1, dtype=np.int64)
    if ok.any():
        with np.errstate(all="ignore"):
            e, z = sq_errors(to32(Rh[ok], th[ok]), rows, camera)
        count[ok] = ((z > 0) & (e < t2_of(threshold))).sum(1)
    out = dict(hyp_count=count, best=-1, hyp_mask=np.zeros(n, bool), refit_used=False, R=np.zeros((3, 3)),
               t=np.zeros(3), rms=np.zeros(2), mask=np.zeros(n, bool), band=np.zeros(n, bool))
    if not ok.any():
        return out
    best = int(np.argmax(count))
    R0, t0 = Rh[best].reshape(3, 3), th[best]
    hm = inliers(R0, t0, rows, camera, threshold)
    m = int(hm.sum())
    out.update(best=best, hyp_mask=hm)
    if m == 0:                                       # a best sample without an inlier is no model
        return out
    out.update(R=R0, t=t0, mask=hm, band=near_threshold(R0, t0, rows, camera, threshold))
    R1, t1, c0, c1, _ = refine(R0, t0, rows[hm], camera, refine_iters)
    out["rms"] = np.sqrt(np.array([c0, c0]) / m)
    if refine_iters > 0 and m >= MIN_REFINE_ROWS:
        rm = inliers(R1, t1, rows, camera, threshold)
        if rm.sum() >= m:
            out.update(refit_used=True, R=R1, t=t1, mask=rm, rms=np.sqrt(np.array([c0, c1]) / m),
                       band=near_threshold(R1, t1, rows, camera, threshold))
    return out
