"""RANSAC homography (csrc/ransac.cu) restated in NumPy — TEST INFRASTRUCTURE ONLY.

The sampler, the normalised 4-point DLT and the fp32 scoring follow the kernel operation by
operation: NumPy's element-wise loops round every product and sum separately (no contraction), as
the kernel's __dmul_rn / __dadd_rn and __fmul_rn / __fadd_rn do, and the elimination visits rows and
pivots in the kernel's order.  Hypotheses, per-hypothesis inlier counts and the best index are
therefore bit-identical to the device's.  The refit uses np.linalg.eigh on this module's own normal
matrix (the kernel: fixed-order block reductions and Jacobi), so a refit H agrees to rounding only.
"""

import numpy as np

GOLDEN = np.uint64(0x9E3779B97F4A7C15)
MAX_DRAWS = 32
PIVOT_TOL = 1e-8
SQRT2 = 1.4142135623730951


def splitmix64(seed, k):
    """Output k (0-based, array) of the splitmix64 stream seeded with ``seed``."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (np.asarray(k, dtype=np.uint64) + np.uint64(1)) * GOLDEN
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def sample4(seed, n, hyps):
    """Rows of hypotheses ``hyps`` (array) for a list of n rows -> idx (H,4) int64, ok (H,) bool.
    Draw c of hypothesis h is output h*32 + c; a row already drawn is redrawn; 32 draws at most."""
    hyps = np.asarray(hyps, dtype=np.uint64)
    u = splitmix64(seed, hyps[:, None] * np.uint64(MAX_DRAWS) + np.arange(MAX_DRAWS, dtype=np.uint64)[None])
    vals = (((u >> np.uint64(32)) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
    H = hyps.shape[0]
    idx = np.full((H, 4), -1, dtype=np.int64)
    got = np.zeros(H, dtype=np.int64)
    rows = np.arange(H)
    for c in range(MAX_DRAWS):
        v = vals[:, c]
        take = (got < 4) & ~(idx == v[:, None]).any(axis=1)
        idx[rows[take], got[take]] = v[take]
        got += take
    return idx, got == 4


def _norm4(x, y):
    cx = (((x[:, 0] + x[:, 1]) + x[:, 2]) + x[:, 3]) * 0.25
    cy = (((y[:, 0] + y[:, 1]) + y[:, 2]) + y[:, 3]) * 0.25
    md = None
    for q in range(4):
        dx, dy = x[:, q] - cx, y[:, q] - cy
        d = np.sqrt(dx * dx + dy * dy)
        md = d if md is None else md + d
    md = md * 0.25
    ok = md > 0.0
    s = SQRT2 / np.where(ok, md, 1.0)
    return cx, cy, s, ok


def denormalise(hn, s1, cx1, cy1, s2, cx2, cy2):
    """H = T2^-1 . Hn . T1 scaled to h33 = 1, as the kernel forms it.  hn (H,9) -> (H,9), ok (H,)."""
    tx, ty = (-s1) * cx1, (-s1) * cy1
    m = np.empty_like(hn)
    for r in range(3):
        m[:, 3 * r] = hn[:, 3 * r] * s1
        m[:, 3 * r + 1] = hn[:, 3 * r + 1] * s1
        m[:, 3 * r + 2] = (hn[:, 3 * r] * tx + hn[:, 3 * r + 1] * ty) + hn[:, 3 * r + 2]
    is2 = 1.0 / s2
    out = np.empty_like(hn)
    for c in range(3):
        out[:, c] = is2 * m[:, c] + cx2 * m[:, 6 + c]
        out[:, 3 + c] = is2 * m[:, 3 + c] + cy2 * m[:, 6 + c]
        out[:, 6 + c] = m[:, 6 + c]
    w = out[:, 8].copy()
    ok = np.abs(w) >= PIVOT_TOL
    out[:, :8] = out[:, :8] / np.where(ok, w, 1.0)[:, None]
    out[:, 8] = 1.0
    ok &= np.isfinite(out[:, :8]).all(axis=1)
    return out, ok


def dlt4(q):
    """q (H,4,4) float32 rows (x1,y1,x2,y2) -> H (H,9) float64 with h33 = 1, ok (H,)."""
    q = q.astype(np.float64)
    x1, y1, x2, y2 = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    cx1, cy1, s1, ok1 = _norm4(x1, y1)
    cx2, cy2, s2, ok2 = _norm4(x2, y2)
    n = q.shape[0]
    A = np.zeros((n, 8, 9))
    for k in range(4):
        x, y = (x1[:, k] - cx1) * s1, (y1[:, k] - cy1) * s1
        u, v = (x2[:, k] - cx2) * s2, (y2[:, k] - cy2) * s2
        A[:, 2 * k, 0], A[:, 2 * k, 1], A[:, 2 * k, 2] = x, y, 1.0
        A[:, 2 * k, 6], A[:, 2 * k, 7], A[:, 2 * k, 8] = (-u) * x, (-u) * y, u
        A[:, 2 * k + 1, 3], A[:, 2 * k + 1, 4], A[:, 2 * k + 1, 5] = x, y, 1.0
        A[:, 2 * k + 1, 6], A[:, 2 * k + 1, 7], A[:, 2 * k + 1, 8] = (-v) * x, (-v) * y, v
    ok = ok1 & ok2
    for c in range(8):
        for r in range(c + 1, 8):
            sw = np.abs(A[:, r, c]) > np.abs(A[:, c, c])
            t = A[sw, c, c:].copy()
            A[sw, c, c:] = A[sw, r, c:]
            A[sw, r, c:] = t
        ok &= np.abs(A[:, c, c]) >= PIVOT_TOL
        piv = A[:, c, c]
        for r in range(c + 1, 8):
            f = A[:, r, c] / piv
            A[:, r, c + 1:] = A[:, r, c + 1:] - f[:, None] * A[:, c, c + 1:]
    hn = np.zeros((n, 9))
    hn[:, 8] = 1.0
    for c in range(7, -1, -1):
        acc = A[:, c, 8].copy()
        for k in range(c + 1, 8):
            acc = acc - A[:, c, k] * hn[:, k]
        hn[:, c] = acc / A[:, c, c]
    H, okd = denormalise(hn, s1, cx1, cy1, s2, cx2, cy2)
    return H, ok & okd


def sq_errors(H32, pts):
    """Forward transfer errors in the kernel's fp32 order: H32 (H,9) float32, pts (n,4) float32 -> (H,n)."""
    h = [H32[:, k:k + 1] for k in range(9)]
    x, y, x2, y2 = (pts[None, :, c] for c in range(4))
    u = (h[0] * x + h[1] * y) + h[2]
    v = (h[3] * x + h[4] * y) + h[5]
    w = (h[6] * x + h[7] * y) + h[8]
    iw = np.float32(1.0) / w
    dx = u * iw - x2
    dy = v * iw - y2
    return dx * dx + dy * dy


def t2_of(threshold):
    return np.float32(float(threshold) * float(threshold))


def inliers(H64, pts, threshold):
    """Inlier mask (n,) of one double homography after rounding it to fp32, as the kernel scores."""
    with np.errstate(all="ignore"):
        return sq_errors(np.asarray(H64, dtype=np.float64).reshape(1, 9).astype(np.float32), pts)[0] < t2_of(threshold)


def hypotheses(pts, iters, seed):
    """All hypotheses of one list: (H (iters,9) float64, ok (iters,))."""
    n = pts.shape[0]
    if n < 4:
        return np.zeros((iters, 9)), np.zeros(iters, dtype=bool)
    idx, ok = sample4(seed, n, np.arange(iters))
    q = pts[np.where(ok[:, None], idx, 0)]
    with np.errstate(all="ignore"):
        H, okh = dlt4(q)
    return H, ok & okh


def refit(pts, mask):
    """Least-squares normalised DLT over pts[mask] (smallest eigenvector of the normal matrix)."""
    q = pts[mask].astype(np.float64)
    c1, c2 = q[:, :2].mean(0), q[:, 2:].mean(0)
    md1 = np.sqrt(((q[:, :2] - c1) ** 2).sum(1)).mean()
    md2 = np.sqrt(((q[:, 2:] - c2) ** 2).sum(1)).mean()
    if not (md1 > 0 and md2 > 0):
        return None
    s1, s2 = SQRT2 / md1, SQRT2 / md2
    x, y = (q[:, 0] - c1[0]) * s1, (q[:, 1] - c1[1]) * s1
    u, v = (q[:, 2] - c2[0]) * s2, (q[:, 3] - c2[1]) * s2
    z, o = np.zeros_like(x), np.ones_like(x)
    A = np.concatenate([np.stack([x, y, o, z, z, z, -u * x, -u * y, -u], 1),
                        np.stack([z, z, z, x, y, o, -v * x, -v * y, -v], 1)])
    _, V = np.linalg.eigh(A.T @ A)
    H, ok = denormalise(V[:, 0][None].copy(), s1, c1[0], c1[1], s2, c2[0], c2[1])
    return H[0] if ok[0] else None


def verify(pts, iters=1024, threshold=3.0, seed=0):
    """One match list as correspondences pts (n,4) float32 (x1,y1,x2,y2) in list order -> dict:
    hyp_count (iters,) int (-1 degenerate), best (-1 none), hyp_mask (n,) before the refit,
    refit_used, H (9,) float64 (zeros: no model), mask (n,) final inliers."""
    pts = np.ascontiguousarray(pts, dtype=np.float32).reshape(-1, 4)
    n = pts.shape[0]
    Hh, ok = hypotheses(pts, iters, seed)
    count = np.full(iters, -1, dtype=np.int64)
    if ok.any():
        with np.errstate(all="ignore"):
            e = sq_errors(Hh[ok].astype(np.float32), pts)
        count[ok] = (e < t2_of(threshold)).sum(1)
    out = dict(hyp_count=count, best=-1, hyp_mask=np.zeros(n, dtype=bool), refit_used=False,
               H=np.zeros(9), mask=np.zeros(n, dtype=bool))
    if not ok.any():
        return out
    best = int(np.argmax(count))                     # lowest index among the maxima
    hm = inliers(Hh[best], pts, threshold)
    out.update(best=best, hyp_mask=hm, H=Hh[best], mask=hm)
    if hm.sum() >= 4:
        Hr = refit(pts, hm)
        if Hr is not None:
            rm = inliers(Hr, pts, threshold)
            if rm.sum() >= hm.sum():
                out.update(refit_used=True, H=Hr, mask=rm)
    return out
