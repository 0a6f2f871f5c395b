"""RANSAC fundamental matrix (csrc/ransac.cu, the FModel instantiation) restated in NumPy — TEST
INFRASTRUCTURE ONLY.

Like oracle/geometry.py for the homography, the sampler, the 7-point solve and the fp32 scoring follow
the kernel operation by operation: NumPy's element-wise loops round every product, sum and quotient
separately (no contraction), as the kernel's __dmul_rn / __dadd_rn / __ddiv_rn / __dsqrt_rn and
__fmul_rn / __fadd_rn / __frcp_rn do; the full-pivot elimination, the root finder (critical points by
the quadratic formula, 64 bisection steps per bracket) and the slot order are the kernel's.  Hypotheses,
per-slot inlier counts and the best slot are therefore bit-identical to the device's.  The refit uses
np.linalg.eigh (the kernel: fixed-order block reductions and Jacobi), so a refit F agrees to rounding.

Sample s owns slots 3s, 3s+1, 3s+2: the real roots of det(F2 + lam (F1 - F2)) in the order the root
finder produces them — roots of p(lam) on [-1, 1] ascending, then roots of q(mu) = mu^3 p(1/mu) on
(-1, 1) ascending (mu = 0 is F1 - F2).  Unused slots are degenerate.
"""

import numpy as np

from .geometry import MAX_DRAWS, PIVOT_TOL, SQRT2, splitmix64, t2_of

SAMPLE = 7          # rows per sample
SLOTS = 3           # hypothesis slots per sample (real roots of the cubic)
MIN_FIT = 8         # inliers needed for the 8-point refit
BISECT = 64         # bisection steps per sign-changing bracket


def sample_rows(seed, n, samples, R=SAMPLE):
    """R distinct rows of [0, n) per sample (array) -> idx (S,R) int64, ok (S,) bool.  Draw c of sample s
    is output s*32 + c; a row already drawn is redrawn; 32 draws at most.  R = 4 is geometry.sample4."""
    samples = np.asarray(samples, dtype=np.uint64)
    u = splitmix64(seed, samples[:, None] * np.uint64(MAX_DRAWS) + np.arange(MAX_DRAWS, dtype=np.uint64)[None])
    vals = (((u >> np.uint64(32)) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
    S = samples.shape[0]
    idx = np.full((S, R), -1, dtype=np.int64)
    got = np.zeros(S, dtype=np.int64)
    rows = np.arange(S)
    for c in range(MAX_DRAWS):
        v = vals[:, c]
        take = (got < R) & ~(idx == v[:, None]).any(axis=1)
        idx[rows[take], got[take]] = v[take]
        got += take
    return idx, got == R


def _norm(x, y):
    """Centroid and sqrt(2) / mean distance of the R points in each row of x, y (S,R)."""
    R = x.shape[1]
    sx, sy = x[:, 0], y[:, 0]
    for q in range(1, R):
        sx, sy = sx + x[:, q], sy + y[:, q]
    cx, cy = sx / float(R), sy / float(R)
    md = None
    for q in range(R):
        dx, dy = x[:, q] - cx, y[:, q] - cy
        d = np.sqrt(dx * dx + dy * dy)
        md = d if md is None else md + d
    md = md / float(R)
    ok = md > 0.0
    return cx, cy, SQRT2 / np.where(ok, md, 1.0), ok


def null_basis(A):
    """Gaussian elimination with full pivoting of A (S,7,9): pivot = largest |entry| of the remaining
    submatrix, lowest (row, column) on ties; rows below the pivot are reduced in the columns that have
    not pivoted yet.  The two columns that never pivot, j1 < j2, give f1 (f[j1] = 1, f[j2] = 0) and f2
    by back substitution in fixed order.  ok: every pivot >= 1e-8 in magnitude."""
    S = A.shape[0]
    A = A.copy()
    rows = np.arange(S)
    used = np.zeros((S, 9), dtype=bool)
    piv = np.zeros((S, 7), dtype=np.int64)
    ok = np.ones(S, dtype=bool)
    for r in range(7):
        sub = np.where(used[:, None, :], -1.0, np.abs(A[:, r:, :])).reshape(S, -1)
        flat = sub.argmax(axis=1)
        i, c = r + flat // 9, flat % 9
        t = A[rows, r].copy()
        A[rows, r] = A[rows, i]
        A[rows, i] = t
        used[rows, c] = True
        piv[:, r] = c
        p = A[rows, r, c]
        ok &= np.abs(p) >= PIVOT_TOL
        for i2 in range(r + 1, 7):
            f = A[rows, i2, c] / p
            A[:, i2] = np.where(used, A[:, i2], A[:, i2] - f[:, None] * A[:, r])
    free = np.argsort(used, axis=1, kind="stable")[:, :2]
    basis = []
    for j in (free[:, 0], free[:, 1]):
        f = np.zeros((S, 9))
        f[rows, j] = 1.0
        for r in range(6, -1, -1):
            acc = A[rows, r, j]
            for r2 in range(r + 1, 7):
                acc = acc + A[rows, r, piv[:, r2]] * f[rows, piv[:, r2]]
            f[rows, piv[:, r]] = (-acc) / A[rows, r, piv[:, r]]
        basis.append(f)
    return basis[0], basis[1], ok


def _det3(r0, r1, r2):
    """r0 . (r1 x r2) in fixed order; each argument is a tuple of 3 arrays."""
    k0 = r1[1] * r2[2] - r1[2] * r2[1]
    k1 = r1[2] * r2[0] - r1[0] * r2[2]
    k2 = r1[0] * r2[1] - r1[1] * r2[0]
    return (r0[0] * k0 + r0[1] * k1) + r0[2] * k2


def cubic_coeffs(f1, f2):
    """det(F2 + lam D), D = F1 - F2, as (c3, c2, c1, c0) from the 8 row-mixed determinants."""
    d = f1 - f2
    a = [tuple(f2[:, 3 * r + k] for k in range(3)) for r in range(3)]
    b = [tuple(d[:, 3 * r + k] for k in range(3)) for r in range(3)]
    c0 = _det3(a[0], a[1], a[2])
    c1 = (_det3(b[0], a[1], a[2]) + _det3(a[0], b[1], a[2])) + _det3(a[0], a[1], b[2])
    c2 = (_det3(a[0], b[1], b[2]) + _det3(b[0], a[1], b[2])) + _det3(b[0], b[1], a[2])
    c3 = _det3(b[0], b[1], b[2])
    return c3, c2, c1, c0


def _poly(a3, a2, a1, a0, x):
    return ((a3 * x + a2) * x + a1) * x + a0


def cubic_roots(a3, a2, a1, a0, closed=True):
    """Real roots of a3 x^3 + a2 x^2 + a1 x + a0 on [-1, 1] (closed) or (-1, 1), ascending.
    Arrays (S,) -> candidates (S,7) float64 and valid (S,7).  The interval is split at the real critical
    points (quadratic formula, correctly rounded sqrt); a breakpoint where the polynomial is exactly 0 is
    a root, and each bracket with a strict sign change is bisected 64 times."""
    a3, a2, a1, a0 = (np.asarray(v, dtype=np.float64) for v in (a3, a2, a1, a0))
    S = a3.shape[0]
    lo, hi = np.full(S, -1.0), np.full(S, 1.0)
    t3 = 3.0 * a3
    disc = a2 * a2 - t3 * a1
    quad = (a3 != 0.0) & (disc >= 0.0)
    sq = np.sqrt(np.where(quad, disc, 0.0))
    den = np.where(quad, t3, 1.0)
    r1, r2 = (-a2 - sq) / den, (-a2 + sq) / den
    lin = (a3 == 0.0) & (a2 != 0.0)
    cl = (-a1) / np.where(lin, 2.0 * a2, 1.0)
    cA = np.where(quad, np.where(r1 < r2, r1, r2), cl)
    cB = np.where(r1 < r2, r2, r1)
    hA, hB = quad | lin, quad & (disc > 0.0)
    vA = hA & (cA > lo) & (cA < hi)
    vB = hB & (cB > lo) & (cB < hi)
    pA = np.where(vA, cA, lo)
    pB = np.where(vB, cB, pA)
    pts = np.stack([lo, pA, pB, hi], 1)
    valid = np.stack([np.ones(S, bool), vA, vB, np.ones(S, bool)], 1)
    co = [v[:, None] for v in (a3, a2, a1, a0)]
    G = _poly(*co, pts)
    a, b, ga, gb = pts[:, :3], pts[:, 1:], G[:, :3], G[:, 1:]
    br = ((ga < 0.0) & (gb > 0.0)) | ((ga > 0.0) & (gb < 0.0))
    neg = ga < 0.0
    for _ in range(BISECT):
        m = (a + b) * 0.5
        left = (_poly(*co, m) < 0.0) == neg
        a, b = np.where(left, m, a), np.where(left, b, m)
    mid = (a + b) * 0.5
    zero = valid & (G == 0.0)
    if not closed:
        zero[:, 0] = zero[:, 3] = False
    cand = np.empty((S, 7))
    ok = np.empty((S, 7), dtype=bool)
    cand[:, 0::2], ok[:, 0::2] = pts, zero
    cand[:, 1::2], ok[:, 1::2] = mid, br
    return cand, ok


def denormalise(fn, s1, cx1, cy1, s2, cx2, cy2):
    """F = T2^T Fn T1 (T = [[s,0,-s cx],[0,s,-s cy],[0,0,1]]) scaled to unit Frobenius norm with its
    largest-|entry| element (lowest index on ties) positive.  fn (S,9) -> F (S,9), ok (S,): finite, norm > 0."""
    tx, ty = (-s1) * cx1, (-s1) * cy1
    m = np.empty_like(fn)
    for r in range(3):
        m[:, 3 * r] = fn[:, 3 * r] * s1
        m[:, 3 * r + 1] = fn[:, 3 * r + 1] * s1
        m[:, 3 * r + 2] = (fn[:, 3 * r] * tx + fn[:, 3 * r + 1] * ty) + fn[:, 3 * r + 2]
    ux, uy = (-s2) * cx2, (-s2) * cy2
    F = np.empty_like(fn)
    for c in range(3):
        F[:, c] = s2 * m[:, c]
        F[:, 3 + c] = s2 * m[:, 3 + c]
        F[:, 6 + c] = (ux * m[:, c] + uy * m[:, 3 + c]) + m[:, 6 + c]
    n2 = F[:, 0] * F[:, 0]
    for k in range(1, 9):
        n2 = n2 + F[:, k] * F[:, k]
    nrm = np.sqrt(n2)
    ok = (nrm > 0.0) & np.isfinite(nrm)
    F = F / np.where(ok, nrm, 1.0)[:, None]
    big = np.abs(F).argmax(axis=1)
    F = np.where((F[np.arange(F.shape[0]), big] < 0.0)[:, None], -F, F)
    return F, ok & np.isfinite(F).all(axis=1)


def seven_point(q):
    """q (S,7,4) float32 rows (x1,y1,x2,y2) -> F (S,3,9) float64 per slot, ok (S,3)."""
    q = q.astype(np.float64)
    x1, y1, x2, y2 = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    cx1, cy1, s1, ok1 = _norm(x1, y1)
    cx2, cy2, s2, ok2 = _norm(x2, y2)
    S = q.shape[0]
    x, y = (x1 - cx1[:, None]) * s1[:, None], (y1 - cy1[:, None]) * s1[:, None]
    u, v = (x2 - cx2[:, None]) * s2[:, None], (y2 - cy2[:, None]) * s2[:, None]
    A = np.stack([u * x, u * y, u, v * x, v * y, v, x, y, np.ones_like(x)], 2)
    f1, f2, okp = null_basis(A)
    ok = ok1 & ok2 & okp
    c3, c2, c1, c0 = cubic_coeffs(f1, f2)
    lam, okl = cubic_roots(c3, c2, c1, c0, closed=True)
    mu, okm = cubic_roots(c0, c1, c2, c3, closed=False)
    d = f1 - f2
    cand = np.concatenate([f2[:, None] + lam[:, :, None] * d[:, None],          # F2 + lam D
                           mu[:, :, None] * f2[:, None] + d[:, None]], 1)       # mu F2 + D
    cok = np.concatenate([okl, okm], 1) & ok[:, None]
    F = np.zeros((S, SLOTS, 9))
    okF = np.zeros((S, SLOTS), dtype=bool)
    slot = np.cumsum(cok, axis=1) - 1
    s1b, cx1b, cy1b, s2b, cx2b, cy2b = (np.repeat(v, cand.shape[1]) for v in (s1, cx1, cy1, s2, cx2, cy2))
    Fd, okd = denormalise(cand.reshape(-1, 9), s1b, cx1b, cy1b, s2b, cx2b, cy2b)
    Fd, okd = Fd.reshape(S, -1, 9), okd.reshape(S, -1)
    for k in range(cand.shape[1]):
        take = cok[:, k] & (slot[:, k] < SLOTS)
        rows = np.nonzero(take)[0]
        F[rows, slot[rows, k]] = Fd[rows, k]
        okF[rows, slot[rows, k]] = okd[rows, k]
    return F, okF


def hypotheses(pts, iters, seed):
    """All slots of one list: (F (3*iters,9) float64, ok (3*iters,))."""
    n = pts.shape[0]
    if n < SAMPLE:
        return np.zeros((SLOTS * iters, 9)), np.zeros(SLOTS * iters, dtype=bool)
    idx, ok = sample_rows(seed, n, np.arange(iters))
    q = pts[np.where(ok[:, None], idx, 0)]
    with np.errstate(all="ignore"):
        F, okF = seven_point(q)
    return F.reshape(-1, 9), (okF & ok[:, None]).reshape(-1)


def sq_errors(F32, pts):
    """Squared distances of each point to the epipolar line of the other, in the kernel's fp32 order:
    F32 (H,9) float32, pts (n,4) float32 -> e1 (image 1), e2 (image 2), each (H,n)."""
    f = [F32[:, k:k + 1] for k in range(9)]
    x1, y1, x2, y2 = (pts[None, :, c] for c in range(4))
    one = np.float32(1.0)
    a2 = (f[0] * x1 + f[1] * y1) + f[2]
    b2 = (f[3] * x1 + f[4] * y1) + f[5]
    c2 = (f[6] * x1 + f[7] * y1) + f[8]
    d2 = (x2 * a2 + y2 * b2) + c2
    e2 = (d2 * d2) * (one / (a2 * a2 + b2 * b2))
    a1 = (f[0] * x2 + f[3] * y2) + f[6]
    b1 = (f[1] * x2 + f[4] * y2) + f[7]
    c1 = (f[2] * x2 + f[5] * y2) + f[8]
    d1 = (x1 * a1 + y1 * b1) + c1
    e1 = (d1 * d1) * (one / (a1 * a1 + b1 * b1))
    return e1, e2


def inlier_counts(F32, pts, threshold, chunk=512):
    t2 = t2_of(threshold)
    out = np.empty(F32.shape[0], dtype=np.int64)
    with np.errstate(all="ignore"):
        for h0 in range(0, F32.shape[0], chunk):
            e1, e2 = sq_errors(F32[h0:h0 + chunk], pts)
            out[h0:h0 + chunk] = ((e1 < t2) & (e2 < t2)).sum(1)
    return out


def inliers(F64, pts, threshold):
    """Inlier mask (n,) of one double F after rounding it to fp32, as the kernel scores: both squared
    distances < t^2 (a NaN distance is an outlier)."""
    t2 = t2_of(threshold)
    with np.errstate(all="ignore"):
        e1, e2 = sq_errors(np.asarray(F64, dtype=np.float64).reshape(1, 9).astype(np.float32), pts)
    return (e1[0] < t2) & (e2[0] < t2)


def refit(pts, mask):
    """Normalised 8-point least squares over pts[mask]: smallest eigenvector of the 9x9 normal matrix,
    rank 2 as Fn - (Fn v3) v3^T (v3: smallest eigenvector of Fn^T Fn), then denormalise, unit norm and
    sign rule.  -> F (9,) or None."""
    q = pts[mask].astype(np.float64)
    c1, c2 = q[:, :2].mean(0), q[:, 2:].mean(0)
    md1 = np.sqrt(((q[:, :2] - c1) ** 2).sum(1)).mean()
    md2 = np.sqrt(((q[:, 2:] - c2) ** 2).sum(1)).mean()
    if not (md1 > 0 and md2 > 0):
        return None
    s1, s2 = SQRT2 / md1, SQRT2 / md2
    x, y = (q[:, 0] - c1[0]) * s1, (q[:, 1] - c1[1]) * s1
    u, v = (q[:, 2] - c2[0]) * s2, (q[:, 3] - c2[1]) * s2
    A = np.stack([u * x, u * y, u, v * x, v * y, v, x, y, np.ones_like(x)], 1)
    _, V = np.linalg.eigh(A.T @ A)
    Fn = V[:, 0].reshape(3, 3)
    _, W = np.linalg.eigh(Fn.T @ Fn)
    v3 = W[:, 0]
    Fr = Fn - np.outer(Fn @ v3, v3)
    F, ok = denormalise(Fr.reshape(1, 9), np.float64(s1), c1[0], c1[1], np.float64(s2), c2[0], c2[1])
    return F[0] if ok[0] else None


def verify_fundamental(pts, iters=1024, threshold=3.0, seed=0):
    """One match list as correspondences pts (n,4) float32 (x1,y1,x2,y2) in list order -> dict with the
    keys of geometry.verify: hyp_count (3*iters,) int (-1 degenerate), best slot (-1 none), hyp_mask (n,)
    before the refit, refit_used, H (9,) float64 — here the fundamental matrix, x2^T F x1 = 0, unit norm
    (zeros: no model) — and mask (n,) final inliers."""
    pts = np.ascontiguousarray(pts, dtype=np.float32).reshape(-1, 4)
    n = pts.shape[0]
    Fh, ok = hypotheses(pts, iters, seed)
    count = np.full(SLOTS * iters, -1, dtype=np.int64)
    if ok.any():
        count[ok] = inlier_counts(Fh[ok].astype(np.float32), pts, threshold)
    out = dict(hyp_count=count, best=-1, hyp_mask=np.zeros(n, dtype=bool), refit_used=False,
               H=np.zeros(9), mask=np.zeros(n, dtype=bool))
    if not ok.any():
        return out
    best = int(np.argmax(count))                     # lowest slot among the maxima
    hm = inliers(Fh[best], pts, threshold)
    out.update(best=best, hyp_mask=hm, H=Fh[best], mask=hm)
    if hm.sum() >= MIN_FIT:
        Fr = refit(pts, hm)
        if Fr is not None:
            rm = inliers(Fr, pts, threshold)
            if rm.sum() >= hm.sum():
                out.update(refit_used=True, H=Fr, mask=rm)
    return out


def epipolar_distance(F, pts):
    """Double-precision max(d1, d2) (px) of each row to the epipolar lines of F (9,) — for comparisons."""
    F = np.asarray(F, dtype=np.float64).reshape(3, 3)
    q = np.asarray(pts, dtype=np.float64)
    x1 = np.concatenate([q[:, :2], np.ones((q.shape[0], 1))], 1)
    x2 = np.concatenate([q[:, 2:], np.ones((q.shape[0], 1))], 1)
    l2, l1 = x1 @ F.T, x2 @ F
    num = np.abs((x2 * l2).sum(1))
    with np.errstate(all="ignore"):
        return np.maximum(num / np.hypot(l2[:, 0], l2[:, 1]), num / np.hypot(l1[:, 0], l1[:, 1]))
