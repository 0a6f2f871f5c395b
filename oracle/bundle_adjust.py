"""Sliding-window bundle adjustment (csrc/bundle_adjust.cu) and the window bookkeeping of geometry.py
(window_tracks, window_map) restated — TEST INFRASTRUCTURE ONLY.

``track_links`` restates the provenance geometry.track_and_map(..., want_links=True) returns, from the dict of
oracle/triangulate.py's track_and_map.  ``window_tracks`` / ``window_map`` follow the rules of their device
versions with plain loops over keypoints.
``bundle_adjust`` follows the kernel in NumPy float64: the used set, the Huber weights, per-track sums in
ascending frame order, every sum over tracks in ascending track order (``_seq``: np.cumsum adds in order),
the 3x3 and the reduced-system Cholesky in lm_solve's order, the damping schedule and the depth check.  NumPy
rounds every element-wise operation separately, as the kernel's __dmul_rn / __dadd_rn / __ddiv_rn /
__dsqrt_rn do; only Rodrigues' sin / cos may differ in the last bit.
"""

import math

import numpy as np

LM_LAMBDA0 = 1e-3
LM_LAMBDA_STEP = 10.0


# ---------------------------------------------------------------------------- window bookkeeping
def track_links(point_map, rows, step):
    """One list: point_map (Ka,3) of frame a, rows (n,2), ``step`` = oracle/triangulate.track_and_map's dict for
    them -> (link (Kb,) int32, born (Kb,) bool).  For a keypoint j with a point in step["next_map"], link[j] is
    the frame-a keypoint of the lowest PnP-inlier row with j (born 0: carried), or else of the lowest kept
    triangulation row with j (born 1); -1 and 0 elsewhere."""
    rows = np.asarray(rows).reshape(-1, 2)
    nxt = step["next_map"]
    Ka, Kb = len(point_map), len(nxt)
    i = rows[:, 0]
    has = (i >= 0) & (i < Ka)
    has[has] = np.isfinite(point_map[i[has]]).all(1)
    wr = rows[has]                                      # the rows that entered the PnP, in order
    fin = np.isfinite(nxt).all(1)
    link = np.full(Kb, -1, np.int32)
    born = np.zeros(Kb, bool)
    sources = [(wr, step["pnp"]["mask"], False)]
    if step["tri"] is not None:
        sources.insert(0, (rows, step["tri"]["mask"], True))
    for src, keep, b in sources:                        # triangulated first: carried rows override them
        for k in range(len(src) - 1, -1, -1):           # the lowest row wins
            j = int(src[k, 1])
            if keep[k] and 0 <= j < Kb and fin[j]:
                link[j], born[j] = src[k, 0], b
    return link, born


def window_tracks(maps, links, born, R, t):
    """One window: maps (W,K,3), links / born (W-1,K), R (W,3,3), t (W,3) -> dict(obs (N,W) int32,
    points (N,3) float32, count, track_of (W,K) int32), N = W*K."""
    maps = np.asarray(maps, np.float32)
    W, K = maps.shape[:2]
    N = W * K
    fin = np.isfinite(maps).all(-1)
    root = np.full((W, K), -1, np.int64)            # flat root w*K + j of each keypoint's track
    claim = {}                                      # (w, j) -> keypoint of frame w-1 its born track observes
    for w in range(W):
        taken = set()
        for j in range(K):
            if not fin[w, j]:
                continue
            if w == 0:
                root[w, j] = j
                continue
            lk, bn = int(links[w - 1, j]), bool(born[w - 1, j])
            prev = root[w - 1, lk] if 0 <= lk < K else -1
            if not bn and prev >= 0:
                root[w, j] = prev
            else:
                root[w, j] = w * K + j
                if bn and 0 <= lk < K and prev < 0 and lk not in taken:
                    taken.add(lk)
                    claim[(w, j)] = lk
    roots = sorted({int(r) for r in root.reshape(-1) if r >= 0 and root.reshape(-1)[r] == r})
    index = {r: i for i, r in enumerate(roots)}
    track_of = np.where(root >= 0, np.vectorize(lambda r: index.get(int(r), -1))(root), -1).astype(np.int32)
    obs = np.full((N, W), -1, np.int32)
    for w in range(W):
        for j in range(K - 1, -1, -1):
            if track_of[w, j] >= 0:
                obs[track_of[w, j], w] = j
    for (w, j), lk in claim.items():
        obs[track_of[w, j], w - 1] = lk
    pts = np.full((N, 3), np.nan, np.float32)
    for r in roots:
        w, j = divmod(r, K)
        pts[index[r]] = (np.asarray(R[w], np.float64).T @ (maps[w, j].astype(np.float64) - t[w])).astype(np.float32)
    return dict(obs=obs, points=pts, count=len(roots), track_of=track_of)


def window_map(track_of, points, R, t, obs=None, mask=None):
    """One window: -> (W,K,3) float32, R_w X + t_w of the track of (w, j), NaN where there is none or where the
    keypoint is an observation with mask 0 of a track with at least two observations."""
    W, K = track_of.shape
    out = np.full((W, K, 3), np.nan, np.float32)
    for w in range(W):
        for j in range(K):
            n = int(track_of[w, j])
            if n < 0:
                continue
            if mask is not None and obs[n, w] == j and not mask[n, w] and (obs[n] >= 0).sum() >= 2:
                continue
            out[w, j] = (np.asarray(R[w], np.float64) @ points[n].astype(np.float64) + t[w]).astype(np.float32)
    return out


# ---------------------------------------------------------------------------- the solver
def _seq(a):
    """Sum over axis 0 in ascending order (0.0 for an empty axis)."""
    return np.cumsum(a, axis=0)[-1] if len(a) else np.zeros(a.shape[1:])


def _dot3(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _project(P, X, uv, camera, jac=False):
    """P (W,12) R row-major, t; X (n,3); uv (n,W,2) -> res (n,W,2), z (n,W)[, Jp (n,W,2,6), Jx (n,W,2,3)]."""
    fx, fy, cx, cy = camera
    Xb = X[:, None, :]
    rx = [_dot3(P[None, :, 3 * i:3 * i + 3], Xb) for i in range(3)]
    xc, yc, zc = rx[0] + P[None, :, 9], rx[1] + P[None, :, 10], rx[2] + P[None, :, 11]
    iz = 1.0 / zc
    pu, pv = xc * iz, yc * iz
    res = np.stack([(fx * pu + cx) - uv[..., 0], (fy * pv + cy) - uv[..., 1]], -1)
    if not jac:
        return res, zc
    zero = np.zeros_like(iz)
    gu = np.stack([fx * iz, zero, -((fx * pu) * iz)], -1)
    gv = np.stack([zero, fy * iz, -((fy * pv) * iz)], -1)
    cols = [np.stack([zero, -rx[2], rx[1]], -1), np.stack([rx[2], zero, -rx[0]], -1),
            np.stack([-rx[1], rx[0], zero], -1)]
    Jp = np.stack([np.stack([_dot3(g, cl) for cl in cols] + [g[..., 0], g[..., 1], g[..., 2]], -1)
                   for g in (gu, gv)], -2)
    Rc = [np.broadcast_to(P[None, :, [j, 3 + j, 6 + j]], gu.shape) for j in range(3)]
    Jx = np.stack([np.stack([_dot3(g, Rc[j]) for j in range(3)], -1) for g in (gu, gv)], -2)
    return res, zc, Jp, Jx


def _rho(s, d):
    d2 = d * d
    with np.errstate(invalid="ignore"):
        return np.where(s <= d2, s, (2.0 * d) * np.sqrt(s) - d2)


def _frames(v, use):
    """Per-track sum over frames in ascending order of v (n,W,...) where use (n,W)."""
    acc = np.zeros((v.shape[0],) + v.shape[2:])
    for w in range(v.shape[1]):
        u = use[:, w].reshape((-1,) + (1,) * (v.ndim - 2))
        acc = acc + np.where(u, v[:, w], 0.0)
    return acc


def _chol3(V, lam):
    """V (n,6) upper -> L (n,6) lower (00 10 11 20 21 22), positive definite (n,)."""
    a00, a11, a22 = V[:, 0] + lam * V[:, 0], V[:, 3] + lam * V[:, 3], V[:, 5] + lam * V[:, 5]
    with np.errstate(all="ignore"):
        L0 = np.sqrt(a00)
        L1 = V[:, 1] / L0
        L3 = V[:, 2] / L0
        d1 = a11 - L1 * L1
        L2 = np.sqrt(d1)
        L4 = (V[:, 4] - L3 * L1) / L2
        d2 = (a22 - L3 * L3) - L4 * L4
        L5 = np.sqrt(d2)
    return np.stack([L0, L1, L2, L3, L4, L5], 1), (a00 > 0.0) & (d1 > 0.0) & (d2 > 0.0)


def _fwd3(L, b):
    L = L.reshape(L.shape[:1] + (1,) * (b.ndim - 2) + (6,))
    y0 = b[..., 0] / L[..., 0]
    y1 = (b[..., 1] - L[..., 1] * y0) / L[..., 2]
    y2 = ((b[..., 2] - L[..., 3] * y0) - L[..., 4] * y1) / L[..., 5]
    return np.stack([y0, y1, y2], -1)


def _bwd3(L, h):
    x2 = h[:, 2] / L[:, 5]
    x1 = (h[:, 1] - L[:, 4] * x2) / L[:, 2]
    x0 = ((h[:, 0] - L[:, 1] * x1) - L[:, 3] * x2) / L[:, 0]
    return np.stack([x0, x1, x2], 1)


def _exp(w):
    """geometry.cuh's rodrigues."""
    th = math.sqrt(float((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]))
    X = np.eye(3)
    if th > 0.0:
        k = w / th
        K = np.array([[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]])
        K2 = np.array([[(K[i, 0] * K[0, j] + K[i, 1] * K[1, j]) + K[i, 2] * K[2, j] for j in range(3)] for i in range(3)])
        X = (X + math.sin(th) * K) + (1.0 - math.cos(th)) * K2
    return X


def _mat3(A, B):
    return np.array([[(A[i, 0] * B[0, j] + A[i, 1] * B[1, j]) + A[i, 2] * B[2, j] for j in range(3)] for i in range(3)])


def _cholesky_solve(S, v):
    """lm_solve's Cholesky of S (n,n) and the solve S x = v -> x, or None (not positive definite or not finite)."""
    n = len(v)
    Lc = np.zeros((n, n))
    for j in range(n):
        d = S[j, j]
        for k in range(j):
            d = d - Lc[j, k] * Lc[j, k]
        if not d > 0.0:
            return None
        Lc[j, j] = math.sqrt(d)
        for i in range(j + 1, n):
            s = S[i, j]
            for k in range(j):
                s = s - Lc[i, k] * Lc[j, k]
            Lc[i, j] = s / Lc[j, j]
    x = np.zeros(n)
    for i in range(n):
        s = v[i]
        for k in range(i):
            s = s - Lc[i, k] * x[k]
        x[i] = s / Lc[i, i]
    for i in range(n - 1, -1, -1):
        s = x[i]
        for k in range(i + 1, n):
            s = s - Lc[k, i] * x[k]
        x[i] = s / Lc[i, i]
    return x if np.isfinite(x).all() else None


def bundle_adjust(kpts, frame_index, obs, points, count, R, t, camera, fixed=2, huber=3.0, threshold=3.0,
                  refine_iters=10):
    """One window: kpts (F,K,2) float32, frame_index (W,), obs (N,W), points (N,3) float32, count, R (W,3,3),
    t (W,3) -> dict(R, t, points (N,3) float32, rms (2,), accepted, mask (N,W) bool, used (N,W) bool, cost0,
    cost, s (N,W) final squared errors)."""
    kpts = np.asarray(kpts, np.float32)
    F, K = kpts.shape[:2]
    fi = np.asarray(frame_index).reshape(-1)
    W = len(fi)
    obs = np.asarray(obs).reshape(-1, W)
    N = len(obs)
    pts32 = np.asarray(points, np.float32).reshape(N, 3)
    P = np.concatenate([np.asarray(R, np.float64).reshape(W, 9), np.asarray(t, np.float64).reshape(W, 3)], 1)
    cnt = min(max(int(count), 0), N)
    out = dict(R=P[:, :9].reshape(W, 3, 3).copy(), t=P[:, 9:].copy(), points=pts32.copy(), rms=np.zeros(2),
               accepted=0, mask=np.zeros((N, W), bool), used=np.zeros((N, W), bool), cost0=0.0, cost=0.0,
               s=np.zeros((N, W)))
    if not (np.isfinite(P).all() and all(P[w, :9].any() for w in range(W))):
        return out
    hd = float(huber)
    nf = W - fixed
    NPf = 6 * nf
    # ---- used set
    X = pts32[:cnt].astype(np.float64)
    k = obs[:cnt].astype(np.int64)
    okk = (k >= 0) & (k < K) & (fi[None] >= 0) & (fi[None] < F)
    uv = np.zeros((cnt, W, 2))
    sl, kk = np.clip(fi, 0, F - 1), np.clip(k, 0, K - 1)
    uv[:] = kpts[sl[None, :].repeat(cnt, 0), kk].astype(np.float64)
    with np.errstate(all="ignore"):
        ok = okk & np.isfinite(uv).all(-1) & np.isfinite(X).all(-1, keepdims=True)
        _, z = _project(P, np.where(np.isfinite(X), X, 0.0), uv, camera)
        ok &= z > 0.0
    tr = ok.sum(1) >= 2
    idx = np.flatnonzero(tr)                           # used tracks, ascending
    use = ok[idx]
    out["used"][idx] = use
    if len(idx) == 0:
        return out
    X, uv = X[idx], uv[idx]
    nobs = float(use.sum())

    def cost_of(P_, X_):
        with np.errstate(all="ignore"):
            res, z_ = _project(P_, X_, uv, camera)
        s = res[..., 0] * res[..., 0] + res[..., 1] * res[..., 1]
        return _seq(_frames(_rho(s, hd), use)), s, z_

    cost, s0, _ = cost_of(P, X)
    ss0 = _seq(_frames(s0, use))
    cost0 = cost

    def linearise(P_, X_):
        res, _, Jp, Jx = _project(P_, X_, uv, camera, jac=True)
        s = res[..., 0] * res[..., 0] + res[..., 1] * res[..., 1]
        with np.errstate(divide="ignore"):
            wt = np.minimum(1.0, hd / np.sqrt(s))
        wJp, wJx = wt[..., None, None] * Jp, wt[..., None, None] * Jx
        Vw = np.stack([wJx[..., 0, i] * Jx[..., 0, j] + wJx[..., 1, i] * Jx[..., 1, j]
                       for i in range(3) for j in range(i, 3)], -1)
        bw = np.stack([wJx[..., 0, i] * res[..., 0] + wJx[..., 1, i] * res[..., 1] for i in range(3)], -1)
        Uw = np.stack([wJp[..., 0, i] * Jp[..., 0, j] + wJp[..., 1, i] * Jp[..., 1, j]
                       for i in range(6) for j in range(i, 6)], -1)
        bpw = np.stack([wJp[..., 0, i] * res[..., 0] + wJp[..., 1, i] * res[..., 1] for i in range(6)], -1)
        Ww = np.stack([np.stack([wJp[..., 0, a] * Jx[..., 0, q] + wJp[..., 1, a] * Jx[..., 1, q] for q in range(3)], -1)
                       for a in range(6)], -2)                                # (n,W,6,3)
        return dict(V=_frames(Vw, use), bx=_frames(bw, use), U=Uw, bp=bpw, W=Ww)

    iu = [(i, j) for i in range(6) for j in range(i, 6)]
    accepted = 0
    if refine_iters > 0:
        lin = linearise(P, X)

        def pose_sums(lin):
            U = np.zeros((max(nf, 0), 21))
            bp = np.zeros((max(nf, 0), 6))
            for f in range(nf):
                w = fixed + f
                U[f] = _seq(np.where(use[:, w, None], lin["U"][:, w], 0.0))
                bp[f] = _seq(np.where(use[:, w, None], lin["bp"][:, w], 0.0))
            return U, bp

        U, bp = pose_sums(lin)
        d = 0.0
        for i in range(NPf):
            d = d + U[i // 6, iu.index((i % 6, i % 6))]
        V = lin["V"]
        d = d + _seq((V[:, 0] + V[:, 3]) + V[:, 5])
        lam = LM_LAMBDA0 * (d / (float(NPf) + 3.0 * len(idx)))
        for it in range(refine_iters):
            L, pd = _chol3(lin["V"], lam)
            x = None
            if pd.all():
                g = _fwd3(L, lin["bx"])
                Z = np.zeros((len(idx), NPf, 3))
                for f in range(nf):
                    w = fixed + f
                    Zw = _fwd3(L, lin["W"][:, w])                               # (n,6,3)
                    Z[:, 6 * f:6 * f + 6] = np.where(use[:, w, None, None], Zw, 0.0)
                A = _seq(_dot3(Z[:, :, None, :], Z[:, None, :, :]))
                Ag = _seq(_dot3(Z, g[:, None, :]))
                S = np.zeros((NPf, NPf))
                for i in range(NPf):
                    for j in range(i, NPf):
                        u = 0.0
                        if i // 6 == j // 6:
                            u = U[i // 6, iu.index((i % 6, j % 6))]
                            if i == j:
                                u = u + lam * u
                        S[j, i] = S[i, j] = u - A[i, j]
                v = np.array([Ag[i] - bp[i // 6, i % 6] for i in range(NPf)])
                x = _cholesky_solve(S, v) if NPf else np.zeros(0)
            accept = False
            if x is not None:
                Pn = P.copy()
                for f in range(nf):
                    w = fixed + f
                    E = _exp(x[6 * f:6 * f + 3])
                    Pn[w, :9] = _mat3(E, P[w, :9].reshape(3, 3)).reshape(9)
                    Pn[w, 9:] = P[w, 9:] + x[6 * f + 3:6 * f + 6]
                ql = np.zeros((len(idx), W, 3))
                for f in range(nf):
                    w = fixed + f
                    Zw = _fwd3(L, lin["W"][:, w])
                    q = np.zeros((len(idx), 3))
                    for a in range(6):
                        q = q + Zw[:, a] * x[6 * f + a]
                    ql[:, w] = np.where(use[:, w, None], q, 0.0)
                h = g + _frames(ql, np.ones_like(use))
                Xc = X - _bwd3(L, h)
                c, _, zc = cost_of(Pn, Xc)
                behind = bool((use & ~(zc > 0.0)).any())
                accept = not behind and c < cost
            if accept:
                P, X, cost = Pn, Xc, c
                lam = lam / LM_LAMBDA_STEP
                accepted += 1
                if it + 1 < refine_iters:
                    lin = linearise(P, X)
                    U, bp = pose_sums(lin)
            else:
                lam = lam * LM_LAMBDA_STEP
    _, s1, _ = cost_of(P, X)
    ss1 = _seq(_frames(s1, use))
    out["R"], out["t"] = P[:, :9].reshape(W, 3, 3).copy(), P[:, 9:].copy()
    out["points"][idx] = X.astype(np.float32)
    out["rms"] = np.array([math.sqrt(ss0 / nobs), math.sqrt(ss1 / nobs)])
    out["accepted"] = accepted
    out["mask"][idx] = use & (s1 < threshold * threshold)
    out["s"][idx] = np.where(use, s1, 0.0)
    out.update(cost0=float(cost0), cost=float(cost))
    return out
