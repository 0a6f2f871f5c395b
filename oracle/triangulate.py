"""Triangulation of a match list under a known relative pose (csrc/triangulate.cu) restated in NumPy float64,
and the tracking-with-map-growth step built on it (geometry.track_and_map) — TEST INFRASTRUCTURE ONLY.

Every row follows the kernel's thread operation by operation: the rays and midpoint of oracle/pose.py (the
kernel's geometry.cuh midpoint), the per-row Levenberg-Marquardt on X with the kernel's accumulation order,
3x3 Cholesky and damping schedule, and the gates.  NumPy rounds every element-wise product, sum, quotient
and square root separately, as the kernel's __dmul_rn / __dadd_rn / __ddiv_rn / __dsqrt_rn do, so points and
masks agree bit for bit with the device.  The rows are processed together, each with its own LM state.

``track_and_map`` composes oracle/pnp.py's RANSAC P3P with this triangulation, rounding points to fp32 where
the device stores them.
"""

import math

import numpy as np

from . import pnp as op
from . import pose as opose

NP = 3
LM_LAMBDA0 = 1e-3
LM_LAMBDA_STEP = 10.0


def _dot3(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def residuals(R, t, X, q, camera, jac=False):
    """Pixel residuals (n,4) (u_a, v_a, u_b, v_b) of X (n,3) against q (n,4), depths (n,2), and with ``jac``
    the Jacobian (n,4,3) d res / d X."""
    fx, fy, cx, cy = camera
    Y = np.stack([_dot3(R[i][None], X) + t[i] for i in range(3)], 1)
    res, z, J = [], [], []
    for v, V in enumerate((X, Y)):
        iz = 1.0 / V[:, 2]
        pu, pv = V[:, 0] * iz, V[:, 1] * iz
        z.append(V[:, 2])
        res += [(fx * pu + cx) - q[:, 2 * v], (fy * pv + cy) - q[:, 2 * v + 1]]
        if jac:
            zero = np.zeros_like(iz)
            gu = np.stack([fx * iz, zero, -((fx * pu) * iz)], 1)
            gv = np.stack([zero, fy * iz, -((fy * pv) * iz)], 1)
            if v == 0:
                J += [gu, gv]
            else:
                J += [np.stack([_dot3(g, R[:, k][None]) for k in range(3)], 1) for g in (gu, gv)]
    return np.stack(res, 1), np.stack(z, 1), (np.stack(J, 1) if jac else None)


def linearise(R, t, X, q, camera):
    """lm_add's accumulators (n,10): J^T J upper triangle, J^T r, r^T r, in the kernel's order."""
    r, _, J = residuals(R, t, X, q, camera, jac=True)
    acc = np.zeros((len(X), 10))
    for e in range(4):
        c = 0
        for i in range(NP):
            for k in range(i, NP):
                acc[:, c] = acc[:, c] + J[:, e, i] * J[:, e, k]
                c += 1
        for i in range(NP):
            acc[:, 6 + i] = acc[:, 6 + i] + J[:, e, i] * r[:, e]
        acc[:, 9] = acc[:, 9] + r[:, e] * r[:, e]
    return acc


def lambda0(acc):
    d = ((0.0 + acc[:, 0]) + acc[:, 3]) + acc[:, 5]
    return LM_LAMBDA0 * (d / float(NP))


def solve(acc, lam):
    """geometry.cuh's lm_solve<3> per row -> x (n,3), ok (n,)."""
    n = len(acc)
    A = [[None] * NP for _ in range(NP)]
    c = 0
    for i in range(NP):
        for j in range(i, NP):
            A[i][j] = A[j][i] = acc[:, c]
            c += 1
    for i in range(NP):
        A[i][i] = A[i][i] + lam * A[i][i]
    L = [[np.zeros(n)] * NP for _ in range(NP)]
    ok = np.ones(n, bool)
    for j in range(NP):
        d = A[j][j]
        for k in range(j):
            d = d - L[j][k] * L[j][k]
        ok &= d > 0.0
        L[j][j] = np.sqrt(np.where(d > 0.0, d, 1.0))
        for i in range(j + 1, NP):
            s = A[i][j]
            for k in range(j):
                s = s - L[i][k] * L[j][k]
            L[i][j] = s / L[j][j]
    x = [None] * NP
    for i in range(NP):
        s = -acc[:, 6 + i]
        for k in range(i):
            s = s - L[i][k] * x[k]
        x[i] = s / L[i][i]
    for i in range(NP - 1, -1, -1):
        s = x[i]
        for k in range(i + 1, NP):
            s = s - L[k][i] * x[k]
        x[i] = s / L[i][i]
    x = np.stack(x, 1)
    return x, ok & np.isfinite(x).all(1)


def refine(R, t, X, q, camera, iters, active):
    """refine_iters LM trials on every active row's X -> (X, accepted trials per row)."""
    X = X.copy()
    acc = linearise(R, t, X, q, camera)
    cost = acc[:, 9].copy()
    lam = lambda0(acc)
    accepted = np.zeros(len(X), np.int64)
    for it in range(iters):
        x, ok = solve(acc, lam)
        Xn = X + x
        r, z, _ = residuals(R, t, Xn, q, camera)
        c = (((0.0 + r[:, 0] * r[:, 0]) + r[:, 1] * r[:, 1]) + r[:, 2] * r[:, 2]) + r[:, 3] * r[:, 3]
        acc_ = active & ok & (z[:, 0] > 0.0) & (z[:, 1] > 0.0) & (c < cost)
        X = np.where(acc_[:, None], Xn, X)
        cost = np.where(acc_, c, cost)
        lam = np.where(acc_, lam / LM_LAMBDA_STEP, lam * LM_LAMBDA_STEP)
        accepted += acc_
        if it + 1 < iters and acc_.any():
            acc = np.where(acc_[:, None], linearise(R, t, X, q, camera), acc)
    return X, accepted


def pose_ok(R, t):
    R, t = np.asarray(R, np.float64), np.asarray(t, np.float64)
    return bool(np.isfinite(R).all() and np.isfinite(t).all() and R.any())


def triangulate(pts, R, t, camera, threshold=3.0, min_parallax_deg=1.0, distance_thresh=50.0, refine_iters=10,
                rel=1e-6):
    """One list: pts (n,4) (x1, y1, x2, y2; NaN rows are not usable), R (3,3), t (3,) with x2 ~ R x1 + t ->
    dict(mask (n,) bool, points (n,3) float64 in the camera-1 frame (0 where not kept), midpoint (n,3),
    apart (n,) rays not parallel, accepted (n,) LM trials, band (n,) rows whose decision is within ``rel`` of
    a gate bound, and the gate quantities za, zb, cos, ea, eb)."""
    q = np.asarray(pts, dtype=np.float64).reshape(-1, 4)
    n = len(q)
    R = np.asarray(R, np.float64).reshape(3, 3)
    t = np.asarray(t, np.float64).reshape(3)
    out = dict(mask=np.zeros(n, bool), points=np.zeros((n, 3)), midpoint=np.zeros((n, 3)), apart=np.zeros(n, bool),
               accepted=np.zeros(n, np.int64), band=np.zeros(n, bool))
    if n == 0 or not pose_ok(R, t):
        return out
    max_cos = math.cos(math.radians(min_parallax_deg))
    t2 = threshold * threshold
    f1, f2, usable = opose.rays(q, camera)
    qq = np.where(usable[:, None], q, 0.0)
    with np.errstate(all="ignore"):
        _, X0, info = opose.triangulate(R, t, f1, f2, distance_thresh)
        apart = (info["den"] > info["lim"]) & usable
        X, accepted = (refine(R, t, X0, qq, camera, refine_iters, apart) if refine_iters > 0
                       else (X0, np.zeros(n, np.int64)))
        r, z, _ = residuals(R, t, X, qq, camera)
        cb = -np.array([(R[0, i] * t[0] + R[1, i] * t[1]) + R[2, i] * t[2] for i in range(3)])
        v = X - cb
        cos = _dot3(X, v) / (np.sqrt(_dot3(X, X)) * np.sqrt(_dot3(v, v)))
        ea = r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1]
        eb = r[:, 2] * r[:, 2] + r[:, 3] * r[:, 3]
        za, zb = z[:, 0], z[:, 1]
        keep = (apart & (za > 0.0) & (za < distance_thresh) & (zb > 0.0) & (zb < distance_thresh) &
                (cos <= max_cos) & (ea < t2) & (eb < t2))
        band = ((np.abs(info["den"] - info["lim"]) <= rel * np.abs(info["lim"])) |
                (np.abs(za) <= rel) | (np.abs(za - distance_thresh) <= rel * distance_thresh) |
                (np.abs(zb) <= rel) | (np.abs(zb - distance_thresh) <= rel * distance_thresh) |
                (np.abs(cos - max_cos) <= rel) | (np.abs(ea - t2) <= rel * t2) | (np.abs(eb - t2) <= rel * t2))
    out.update(mask=keep, points=np.where(keep[:, None], X, 0.0), midpoint=X0, apart=apart, accepted=accepted,
               band=band & apart, za=za, zb=zb, cos=cos, ea=ea, eb=eb)
    return out


def carry(X32, R, t):
    """fp32 points of frame a -> fp32 points of frame b, R X + t in float64 (geometry.point_map)."""
    return (np.asarray(X32, np.float32).astype(np.float64) @ np.asarray(R).reshape(3, 3).T +
            np.asarray(t).reshape(3)).astype(np.float32)


def fill(num_keypoints, j, keep, X32, R, t, into=None):
    """point_map for one list: keypoint j[k] of the rows k with keep[k] takes carry(X32[k]) (lowest row wins);
    finite entries of ``into`` are kept.  -> (num_keypoints, 3) float32, NaN where there is no point."""
    M = np.full((num_keypoints, 3), np.nan, np.float32)
    ok = keep & (j >= 0) & (j < num_keypoints)
    if ok.any():
        X2 = carry(X32[ok], R, t)
        jj = j[ok]
        for k in range(len(jj) - 1, -1, -1):
            M[jj[k]] = X2[k]
    if into is not None:
        M = np.where(np.isfinite(into).all(1, keepdims=True), into, M)
    return M


def list_points(kp1, kp2, rows):
    """(n,4) float64 (x1, y1, x2, y2) of list rows (i, j); NaN where an index is out of range."""
    rows = np.asarray(rows).reshape(-1, 2)
    out = np.full((len(rows), 4), np.nan)
    ok = (rows[:, 0] >= 0) & (rows[:, 0] < len(kp1)) & (rows[:, 1] >= 0) & (rows[:, 1] < len(kp2))
    out[ok] = np.concatenate([kp1[rows[ok, 0]], kp2[rows[ok, 1]]], 1)
    return out


def track_and_map(point_map, kp_a, kp_b, rows, camera, threshold=3.0, iters=1024, seed=0, refine_iters=10,
                  min_parallax_deg=1.0, distance_thresh=50.0, tri_refine_iters=10, grow=True):
    """One list of geometry.track_and_map: point_map (Ka,3) float32 of frame a, keypoints kp_a (Ka,2), kp_b
    (Kb,2) float32, rows (n,2) -> dict(R, t, with_points (rows that enter the PnP), pnp (oracle/pnp.py's
    dict), tri (triangulate's dict or None), next_map (Kb,3) float32).  grow=False only carries the PnP
    inliers' points (the map without triangulation)."""
    rows = np.asarray(rows).reshape(-1, 2)
    Ka, Kb = len(point_map), len(kp_b)
    i = rows[:, 0]
    ok_i = (i >= 0) & (i < Ka)
    has = ok_i.copy()
    has[ok_i] = np.isfinite(point_map[i[ok_i]]).all(1)
    wr = rows[has]
    q5 = np.full((len(wr), 5), np.nan, np.float32)
    okj = (wr[:, 1] >= 0) & (wr[:, 1] < Kb)
    q5[:, :3] = point_map[wr[:, 0]]
    q5[okj, 3:] = kp_b[wr[okj, 1]]
    q5[~okj, 3:] = np.nan
    o = op.ransac_pnp(q5, camera, iters=iters, threshold=threshold, seed=seed, refine_iters=refine_iters)
    R, t = o["R"], o["t"]
    carried = fill(Kb, wr[:, 1], o["mask"], q5[:, :3], R, t)
    tri = None
    nxt = carried
    if grow:
        tri = triangulate(list_points(kp_a, kp_b, rows), R, t, camera, threshold=threshold,
                          min_parallax_deg=min_parallax_deg, distance_thresh=distance_thresh,
                          refine_iters=tri_refine_iters)
        nxt = fill(Kb, rows[:, 1], tri["mask"], tri["points"].astype(np.float32), R, t, into=carried)
    if not o["R"].any():
        nxt = np.full((Kb, 3), np.nan, np.float32)
    return dict(R=R, t=t, with_points=int(has.sum()), pnp=o, tri=tri, next_map=nxt)
