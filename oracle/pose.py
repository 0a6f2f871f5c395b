"""Relative pose from a verified match list (csrc/pose.cu) restated in NumPy float64 — TEST
INFRASTRUCTURE ONLY.

The stages follow the kernel in its order: the decomposition of E (Jacobi on E^T E, the same rotation
sequence as geometry.cuh's jacobi_eigen, so eigenvector signs and hence the candidates' order agree), the
per-row rays and midpoint triangulation with the kernel's operation order (NumPy rounds every product, sum
and quotient separately, as the kernel's __dmul_rn / __dadd_rn / __ddiv_rn do), the cheirality counts and
the selection, the Levenberg-Marquardt trials on the signed Sampson distance, and the final cheirality.
The kernel's Jacobi may contract products into FMAs, its reductions run in a fixed tree order, and its
sin / cos are CUDA's, so R, t and the costs agree to rounding rather than bit for bit.
"""

import math

import numpy as np

MIN_REFINE_ROWS = 5
NP = 5


def _dot3(a, b):
    return a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1] + a[..., 2] * b[..., 2]


def _mat3(A, B):
    C = np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            C[i, j] = A[i, 0] * B[0, j] + A[i, 1] * B[1, j] + A[i, 2] * B[2, j]
    return C


def skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def _cross(a, b):
    return np.array([a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]])


def _normalise(v):
    n = math.sqrt(float(_dot3(v, v)))
    if not (n > 0.0) or not math.isfinite(n):
        return None
    return v / n


def jacobi_eigen(A):
    """geometry.cuh's cyclic Jacobi on a symmetric NxN: -> (eigenvalues (N,) = the final diagonal, V with
    column i the eigenvector of eigenvalue i)."""
    A = [list(map(float, r)) for r in np.asarray(A, dtype=np.float64)]
    N = len(A)
    V = [[1.0 if i == j else 0.0 for j in range(N)] for i in range(N)]
    for _ in range(50):
        off = tot = 0.0
        for i in range(N):
            for j in range(N):
                e = A[i][j] * A[i][j]
                tot += e
                if i != j:
                    off += e
        if not (off > 1e-30 * tot):
            break
        for p in range(N - 1):
            for q in range(p + 1, N):
                apq = A[p][q]
                if apq == 0.0:
                    continue
                theta = (A[q][q] - A[p][p]) / (2.0 * apq)
                t = (1.0 if theta >= 0.0 else -1.0) / (abs(theta) + math.sqrt(theta * theta + 1.0))
                c = 1.0 / math.sqrt(t * t + 1.0)
                s = t * c
                for k in range(N):
                    akp, akq = A[k][p], A[k][q]
                    A[k][p], A[k][q] = c * akp - s * akq, s * akp + c * akq
                for k in range(N):
                    apk, aqk = A[p][k], A[q][k]
                    A[p][k], A[q][k] = c * apk - s * aqk, s * apk + c * aqk
                for k in range(N):
                    vkp, vkq = V[k][p], V[k][q]
                    V[k][p], V[k][q] = c * vkp - s * vkq, s * vkp + c * vkq
    return np.array([A[i][i] for i in range(N)]), np.array(V)


def decompose(E):
    """-> (R_a, R_b, t) or None (E zero, not finite, or sigma2 <= 1e-12 sigma1)."""
    e = np.asarray(E, dtype=np.float64).reshape(3, 3)
    n2 = 0.0
    for x in e.reshape(9):
        n2 = n2 + x * x
    nrm = math.sqrt(n2) if n2 >= 0.0 else float("nan")
    if not (nrm > 0.0) or not math.isfinite(nrm):
        return None
    e = e / nrm
    A = np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            A[i, j] = e[0, i] * e[0, j] + e[1, i] * e[1, j] + e[2, i] * e[2, j]
    lam, V = jacobi_eigen(A)
    o = [0, 1, 2]
    for i in range(3):
        for j in range(2, i, -1):
            if lam[o[j]] > lam[o[j - 1]]:
                o[j], o[j - 1] = o[j - 1], o[j]
    s1, s2 = math.sqrt(max(lam[o[0]], 0.0)), math.sqrt(max(lam[o[1]], 0.0))
    if not (s2 > 1e-12 * s1):
        return None
    v = [V[:, o[i]].copy() for i in range(3)]
    if _dot3(v[0], _cross(v[1], v[2])) < 0.0:
        v[2] = -v[2]
    u0 = _normalise(np.array([_dot3(e[k], v[0]) for k in range(3)]))
    if u0 is None:
        return None
    u1 = np.array([_dot3(e[k], v[1]) for k in range(3)])
    u1 = _normalise(u1 - _dot3(u0, u1) * u0)
    if u1 is None:
        return None
    u2 = _cross(u0, u1)
    Ra, Rb = np.empty((3, 3)), np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            x, y, z = u0[i] * v[1][j], u1[i] * v[0][j], u2[i] * v[2][j]
            Ra[i, j] = (x - y) + z
            Rb[i, j] = (y - x) + z
    return Ra, Rb, u2


def candidates(E):
    """The four candidates in the kernel's order, or None."""
    d = decompose(E)
    if d is None:
        return None
    Ra, Rb, t = d
    return [(Ra, t), (Rb, t), (Ra, -t), (Rb, -t)]


def rays(pts, camera):
    """pts (n,4) (x1, y1, x2, y2) -> f1, f2 (n,3) = K^-1 x, usable (n,) bool (all coordinates finite)."""
    fx, fy, cx, cy = camera
    q = np.asarray(pts, dtype=np.float64).reshape(-1, 4)
    usable = np.isfinite(q).all(1)
    q = np.where(usable[:, None], q, 0.0)
    one = np.ones(len(q))
    f1 = np.stack([(q[:, 0] - cx) / fx, (q[:, 1] - cy) / fy, one], 1)
    f2 = np.stack([(q[:, 2] - cx) / fx, (q[:, 3] - cy) / fy, one], 1)
    return f1, f2, usable


def triangulate(R, t, f1, f2, dist):
    """-> good (n,) bool, X (n,3) camera-1 points (|t| = 1), and the row's den, a*c, z1, z2 (for bands)."""
    u = np.stack([_dot3(R[i][None], f1) for i in range(3)], 1)
    a, b, c = _dot3(u, u), _dot3(u, f2), _dot3(f2, f2)
    tt = np.broadcast_to(t, u.shape)
    d, e = _dot3(u, tt), _dot3(f2, tt)
    den = a * c - b * b
    with np.errstate(divide="ignore", invalid="ignore"):
        z1 = (b * e - c * d) / den
    X = np.stack([z1 * f1[:, 0], z1 * f1[:, 1], z1], 1)
    z2 = _dot3(R[2][None], X) + t[2]
    lim = (1e-12 * a) * c
    good = (den > lim) & (z1 > 0.0) & (z1 < dist) & (z2 > 0.0) & (z2 < dist)
    return good, X, dict(den=den, lim=lim, z1=z1, z2=z2)


def near_bound(info, dist, rel=1e-6):
    """Rows whose cheirality decision sits within ``rel`` (relative) of a depth bound or of den's limit."""
    z1, z2, den, lim = info["z1"], info["z2"], info["den"], info["lim"]
    with np.errstate(invalid="ignore"):
        return ((np.abs(z1) <= rel * np.maximum(np.abs(z1), 1.0)) | (np.abs(z1 - dist) <= rel * dist) |
                (np.abs(z2) <= rel * np.maximum(np.abs(z2), 1.0)) | (np.abs(z2 - dist) <= rel * dist) |
                (np.abs(den - lim) <= rel * np.abs(lim)))


def epi_terms(E, f1, f2, camera):
    fx, fy = camera[0], camera[1]
    g = np.stack([_dot3(E[i][None], f1) for i in range(3)], 1)
    h0 = E[0, 0] * f2[:, 0] + E[1, 0] * f2[:, 1] + E[2, 0] * f2[:, 2]
    h1 = E[0, 1] * f2[:, 0] + E[1, 1] * f2[:, 1] + E[2, 1] * f2[:, 2]
    l = np.stack([g[:, 0] / fx, g[:, 1] / fy, h0 / fx, h1 / fy], 1)
    return _dot3(f2, g), l


def _dot4(a, b):
    return a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1] + a[:, 2] * b[:, 2] + a[:, 3] * b[:, 3]


def sampson(E, f1, f2, camera):
    """Signed Sampson distance (px) per row, 0 where the denominator is 0; also l and s = sqrt(s2)."""
    num, l = epi_terms(E, f1, f2, camera)
    s2 = _dot4(l, l)
    s = np.sqrt(s2)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(s2 > 0.0, num / s, 0.0)
    return r, l, s


def basis(t):
    im = 0
    for i in (1, 2):
        if abs(t[i]) < abs(t[im]):
            im = i
    ei = np.zeros(3)
    ei[im] = 1.0
    b1 = _normalise(_cross(t, ei))
    return b1, _cross(t, b1)


def linearise(R, t):
    """-> E = [t]x R, dE (5,3,3) along (w1, w2, w3, d1, d2), B (2,3)."""
    S = skew(t)
    E = _mat3(S, R)
    dE = np.empty((NP, 3, 3))
    for j in range(3):
        ej = np.zeros(3)
        ej[j] = 1.0
        dE[j] = _mat3(_mat3(S, skew(ej)), R)
    b1, b2 = basis(t)
    dE[3], dE[4] = _mat3(skew(b1), R), _mat3(skew(b2), R)
    return E, dE, np.stack([b1, b2])


def residual_jacobian(E, dE, f1, f2, camera):
    """-> r (n,), J (n,5) over the given (usable) rows."""
    r, l, s = sampson(E, f1, f2, camera)
    J = np.zeros((len(r), NP))
    for j in range(NP):
        dnum, dl = epi_terms(dE[j], f1, f2, camera)
        with np.errstate(divide="ignore", invalid="ignore"):
            J[:, j] = np.where(s > 0.0, (dnum - (r * _dot4(l, dl)) / s) / s, 0.0)
    return r, J


def exp_so3(w):
    th = math.sqrt(float(_dot3(w, w)))
    if not th > 0.0:
        return np.eye(3)
    K = skew(np.asarray(w) / th)
    K2 = _mat3(K, K)
    return (np.eye(3) + math.sin(th) * K) + (1.0 - math.cos(th)) * K2


def apply_step(R, t, B, x):
    """Exp(x_w) R, normalise(t + x_d1 b1 + x_d2 b2) (None if t degenerates)."""
    Rn = _mat3(exp_so3(x[:3]), R)
    tn = _normalise((t + x[3] * B[0]) + x[4] * B[1])
    return Rn, tn


def lm_candidate(JtJ, Jtr, lam, R, t, B):
    A = JtJ + lam * np.diag(np.diag(JtJ))
    L = np.zeros((NP, NP))
    for j in range(NP):
        d = A[j, j]
        for k in range(j):
            d = d - L[j, k] * L[j, k]
        if not d > 0.0:
            return None
        L[j, j] = math.sqrt(d)
        for i in range(j + 1, NP):
            s = A[i, j]
            for k in range(j):
                s = s - L[i, k] * L[j, k]
            L[i, j] = s / L[j, j]
    x = np.zeros(NP)
    for i in range(NP):
        s = -Jtr[i]
        for k in range(i):
            s = s - L[i, k] * x[k]
        x[i] = s / L[i, i]
    for i in range(NP - 1, -1, -1):
        s = x[i]
        for k in range(i + 1, NP):
            s = s - L[k, i] * x[k]
        x[i] = s / L[i, i]
    if not np.isfinite(x).all():
        return None
    Rn, tn = apply_step(R, t, B, x)
    return None if tn is None else (Rn, tn)


def refine(R, t, f1, f2, camera, iters):
    """The kernel's LM trials over the usable rows f1, f2 -> (R, t, cost before, cost after, accepted)."""
    E, dE, B = linearise(R, t)
    r, J = residual_jacobian(E, dE, f1, f2, camera)
    cost0 = cost = float(np.sum(r * r))
    JtJ, Jtr = J.T @ J, J.T @ r
    lam = 1e-3 * (float(np.sum(np.diag(JtJ))) / NP)
    accepted = 0
    if iters > 0 and len(f1) >= MIN_REFINE_ROWS:
        for it in range(iters):
            cand = lm_candidate(JtJ, Jtr, lam, R, t, B)
            accept = False
            if cand is not None:
                rn, _, _ = sampson(_mat3(skew(cand[1]), cand[0]), f1, f2, camera)
                c = float(np.sum(rn * rn))
                accept = c < cost
            if accept:
                R, t = cand
                cost, lam = c, lam / 10.0
                accepted += 1
                E, dE, B = linearise(R, t)
                if it + 1 < iters:
                    r, J = residual_jacobian(E, dE, f1, f2, camera)
                    JtJ, Jtr = J.T @ J, J.T @ r
            else:
                lam = lam * 10.0
    return R, t, cost0, cost, accepted


def recover_pose(pts, E, camera, distance_thresh=50.0, refine_iters=10):
    """One list: pts (n,4) (x1, y1, x2, y2; NaN rows are unusable), E (3,3), camera (fx, fy, cx, cy).
    -> dict(have, R, t, cand_good (4,), best, rms (2,), mask (n,) bool, points (n,3), band (n,) bool:
    rows whose final cheirality decision is within 1e-6 of a bound, cand_band (n,) likewise for any
    candidate, accepted LM steps)."""
    pts = np.asarray(pts, dtype=np.float64).reshape(-1, 4)
    n = len(pts)
    f1, f2, usable = rays(pts, camera)
    out = dict(have=False, R=np.zeros((3, 3)), t=np.zeros(3), cand_good=np.zeros(4, np.int64), best=-1,
               rms=np.zeros(2), mask=np.zeros(n, bool), points=np.zeros((n, 3)), band=np.zeros(n, bool),
               cand_band=np.zeros(n, bool), accepted=0)
    cands = candidates(E)
    if cands is None:
        return out
    for c, (R, t) in enumerate(cands):
        good, _, info = triangulate(R, t, f1, f2, distance_thresh)
        out["cand_good"][c] = int((good & usable).sum())
        out["cand_band"] |= near_bound(info, distance_thresh) & usable
    best = int(np.argmax(out["cand_good"]))
    if out["cand_good"][best] == 0:
        return out
    R, t = cands[best]
    R, t, c0, c1, acc = refine(R, t, f1[usable], f2[usable], camera, refine_iters)
    m = int(usable.sum())
    good, X, info = triangulate(R, t, f1, f2, distance_thresh)
    good &= usable
    out.update(have=True, R=R, t=t, best=best, rms=np.sqrt(np.array([c0, c1]) / m), mask=good,
               points=np.where(good[:, None], X, 0.0), band=near_bound(info, distance_thresh) & usable,
               accepted=acc)
    return out
