"""Geometric verification of match lists on the device (csrc/ransac.cu): RANSAC homography, for planar
scenes and rotating cameras, and RANSAC fundamental matrix (the epipolar constraint), for a camera that
translates through a 3-D scene; the relative pose (csrc/pose.cu) of a calibrated camera from the
verified lists: decomposition of E = K^T F K, cheirality, Levenberg-Marquardt refinement of (R, t) and the
triangulated points; and camera tracking (csrc/pnp.cu): the pose of a frame against 3-D points already
triangulated, by RANSAC P3P on 2D-3D match lists with a Levenberg-Marquardt refinement, in the points' units.

Tracking chain — ``recover_pose_device(..., want_mask=True, want_points=True)`` initialises two views (unit
|t|); ``point_map`` moves its points onto the keypoints of the second frame; the next frame's lists from that
frame then pair points with keypoints, and ``solve_pnp_device`` gives that frame's pose in the same units,
so chained poses share one scale (``rows_with_points`` first drops the rows without a point).  ``point_map``
with the PnP's mask and (R, t) carries the points on.  Carrying alone loses points at every frame (a point
survives only while its keypoint stays a PnP inlier), so ``track_and_map`` also triangulates every row of the
step's lists under the PnP pose (``triangulate_device``, csrc/triangulate.cu) and fills the keypoints that
have no carried point with the new points: one batched step of a sequence, in the map's units.

Device API — ``verify_homography_device`` / ``verify_fundamental_device`` take banks of keypoint sets and
the padded lists the matcher produced (``pairs [P,N,2]``, ``pair_scores [P,N]``, ``counts [P]``) and
return, still on the device, one model per pair plus the inlier rows in the same padded format, so every
consumer of match lists (``evaluation.to_match_lists``, ``write_match_lists``,
``pack_match_records``, ``dist.gather_match_lists``) takes the verified lists unchanged and the
estimated ``H`` feeds ``evaluation.ground_truth_matches_device`` directly.

Host API — ``find_homography`` has the arguments and the return shape of ``cv2.findHomography(src,
dst, cv2.RANSAC, thresh)``: ``(H (3,3) float64 or None, mask (n,1) uint8)``; ``find_fundamental`` those
of ``cv2.findFundamentalMat(pts1, pts2, cv2.FM_RANSAC, thresh)``; ``recover_pose`` those of
``cv2.recoverPose(E, pts1, pts2, K, distanceThresh)``; ``solve_pnp_ransac`` those of
``cv2.solvePnPRansac(X, uv, K, None, flags=cv2.SOLVEPNP_P3P)``.
"""

import math

import numpy as np
import torch

from . import ops


def verify_homography_device(kpts1, kpts2, pairs, pair_scores, counts, pair_index=None, num_pairs=None,
                             threshold=3.0, iters=1024, seed=0, want_mask=False, workspace=None):
    """Banks (F1,N,2) / (F2,M,2) and padded lists on device -> (H (P,3,3) float64, pairs, scores, counts
    [, mask (P,L) uint8]) on device.  A pair without a model (fewer than 4 matches, or only degenerate
    samples) has H all zeros and an empty list."""
    return ops.ransac_homography(kpts1, kpts2, pairs, pair_scores, counts, pair_index=pair_index,
                                 num_pairs=num_pairs, threshold=threshold, iters=iters, seed=seed,
                                 want_mask=want_mask, workspace=workspace)


def verify_fundamental_device(kpts1, kpts2, pairs, pair_scores, counts, pair_index=None, num_pairs=None,
                              threshold=3.0, iters=1024, seed=0, want_mask=False, workspace=None):
    """As verify_homography_device, against the epipolar constraint: -> (F (P,3,3) float64, x2^T F x1 = 0,
    unit Frobenius norm, pairs, scores, counts[, mask (P,L) uint8]) on device.  ``iters`` counts 7-point
    samples; a pair without a model (fewer than 7 matches, or only degenerate samples — e.g. an exactly
    planar list) has F all zeros and an empty list."""
    return ops.ransac_fundamental(kpts1, kpts2, pairs, pair_scores, counts, pair_index=pair_index,
                                  num_pairs=num_pairs, threshold=threshold, iters=iters, seed=seed,
                                  want_mask=want_mask, workspace=workspace)


def _host_ransac(fn, src_pts, dst_pts, ransac_thresh, max_iters, seed, what):
    """One host list through fn (ops.ransac_homography / ransac_fundamental) -> (model (3,3) or None,
    mask (n,1) uint8)."""
    if not torch.cuda.is_available():
        raise RuntimeError("sslam_b200 needs a CUDA device (no CPU fallback)")
    src = np.ascontiguousarray(np.asarray(src_pts, dtype=np.float32).reshape(-1, 2))
    dst = np.ascontiguousarray(np.asarray(dst_pts, dtype=np.float32).reshape(-1, 2))
    if src.shape != dst.shape:
        raise ValueError(f"{what} must hold the same number of points")
    n = src.shape[0]
    dev = torch.device("cuda", torch.cuda.current_device())
    L = max(n, 1)
    rows = torch.full((1, L, 2), -1, dtype=torch.int32)
    rows[0, :n, 0] = torch.arange(n, dtype=torch.int32)
    rows[0, :n, 1] = torch.arange(n, dtype=torch.int32)
    k1 = torch.zeros(1, L, 2)                         # at least one row: the C ABI takes no null banks
    k2 = torch.zeros(1, L, 2)
    k1[0, :n], k2[0, :n] = torch.as_tensor(src), torch.as_tensor(dst)
    G, _, _, _, mask = fn(k1.to(dev), k2.to(dev), rows.to(dev), torch.zeros(1, L, device=dev),
                          torch.tensor([n], dtype=torch.int32, device=dev),
                          threshold=ransac_thresh, iters=max_iters, seed=seed, want_mask=True)
    G = G[0].cpu().numpy()
    if not G.any():                                   # no model
        return None, np.zeros((n, 1), dtype=np.uint8)
    return G, mask[0, :n].cpu().numpy().reshape(n, 1)


def find_homography(src_pts, dst_pts, ransac_thresh=3.0, max_iters=1024, seed=0):
    """(n,2) source / destination points -> (H (3,3) float64 with h33 = 1, or None; mask (n,1) uint8).
    n <= 16384 (the list stride limit of sslam_ransac_homography)."""
    return _host_ransac(ops.ransac_homography, src_pts, dst_pts, ransac_thresh, max_iters, seed,
                        "find_homography: src_pts and dst_pts")


def find_fundamental(pts1, pts2, ransac_thresh=3.0, max_iters=1024, seed=0):
    """(n,2) points of image 1 / image 2 -> (F (3,3) float64 with x2^T F x1 = 0, or None; mask (n,1) uint8),
    cv2.findFundamentalMat's return shape.  As cv2 does, F is scaled to F[2,2] = 1 when |F[2,2]| exceeds
    FLT_EPSILON and left at unit Frobenius norm otherwise.  n < 7, or only degenerate samples, gives None
    and an all-zero mask.  ``max_iters`` counts 7-point samples; n <= 16384."""
    F, mask = _host_ransac(ops.ransac_fundamental, pts1, pts2, ransac_thresh, max_iters, seed, "find_fundamental: pts1 and pts2")
    if F is not None and abs(F[2, 2]) > np.finfo(np.float32).eps:
        F = F / F[2, 2]
    return F, mask


def _intrinsics(camera):
    """(fx, fy, cx, cy) or a 3x3 pinhole matrix without skew -> (fx, fy, cx, cy) floats."""
    K = np.asarray(camera, dtype=np.float64)
    if K.shape == (4,):
        return tuple(float(v) for v in K)
    if K.shape != (3, 3):
        raise ValueError("camera must be (fx, fy, cx, cy) or a 3x3 camera matrix")
    if K[0, 1] != 0.0 or K[1, 0] != 0.0 or (K[2] != [0.0, 0.0, 1.0]).any():
        raise ValueError("camera matrix must be [[fx, 0, cx], [0, fy, cy], [0, 0, 1]] (no skew)")
    return float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])


def essential_from_fundamental(F, camera):
    """F (P,3,3) on the device, one camera for both images -> E = K^T F K (P,3,3) float64 on the device.
    Element-wise from the intrinsics (no host copy), so it can be captured in a CUDA graph, and a zero F
    (no model) stays zero."""
    fx, fy, cx, cy = _intrinsics(camera)
    F = F.to(torch.float64)
    FK = torch.stack([fx * F[..., 0], fy * F[..., 1], cx * F[..., 0] + cy * F[..., 1] + F[..., 2]], -1)
    return torch.stack([fx * FK[..., 0, :], fy * FK[..., 1, :], cx * FK[..., 0, :] + cy * FK[..., 1, :] + FK[..., 2, :]],
                       -2)


def recover_pose_device(kpts1, kpts2, E, pairs, scores, counts, camera, pair_index=None, distance_thresh=50.0,
                        refine_iters=10, want_mask=False, want_points=False):
    """Banks, E (P,3,3) float64 and the verified lists on device (usually verify_fundamental_device's) ->
    ops.recover_pose's (R (P,3,3), t (P,3), pairs, scores, counts, cand_good (P,4), rms (P,2)[, mask][,
    points (P,L,3)]) on device.  camera: (fx, fy, cx, cy) or a 3x3 matrix, shared by both images.  A pair
    without a pose (E zero or of rank < 2, or no row in front of both cameras) has R, t all zeros and an
    empty list."""
    fx, fy, cx, cy = _intrinsics(camera)
    return ops.recover_pose(kpts1, kpts2, E, pairs, scores, counts, fx, fy, cx, cy, pair_index=pair_index,
                            distance_thresh=distance_thresh, refine_iters=refine_iters, want_mask=want_mask,
                            want_points=want_points)


def recover_pose(E, pts1, pts2, camera_matrix, distance_thresh=50.0, mask=None, refine_iters=10):
    """cv2.recoverPose(E, pts1, pts2, K, distanceThresh[, mask]) on the device: -> (retval = good rows,
    R (3,3), t (3,1) unit, mask (n,1) uint8, points (4,n) float64 with w = 1: X in the camera-1 frame for
    good rows, (0, 0, 0, 1) elsewhere).  Rows whose input ``mask`` is 0 are left out.  refine_iters = 0
    returns the chosen decomposition candidate, as cv2 does; the default refines it on the Sampson error.
    Without a pose R and t are zeros and retval is 0.  A camera matrix with skew raises ValueError."""
    if not torch.cuda.is_available():
        raise RuntimeError("sslam_b200 needs a CUDA device (no CPU fallback)")
    cam = _intrinsics(camera_matrix)
    p1 = np.ascontiguousarray(np.asarray(pts1, dtype=np.float32).reshape(-1, 2))
    p2 = np.ascontiguousarray(np.asarray(pts2, dtype=np.float32).reshape(-1, 2))
    if p1.shape != p2.shape:
        raise ValueError("recover_pose: pts1 and pts2 must hold the same number of points")
    n = p1.shape[0]
    use = np.ones(n, bool) if mask is None else np.asarray(mask).reshape(-1) != 0
    if use.shape[0] != n:
        raise ValueError("recover_pose: mask must hold one entry per point")
    dev = torch.device("cuda", torch.cuda.current_device())
    L = max(n, 1)
    rows = torch.full((1, L, 2), -1, dtype=torch.int32)
    idx = torch.as_tensor(np.flatnonzero(use).astype(np.int32))
    rows[0, :idx.numel(), 0] = idx
    rows[0, :idx.numel(), 1] = idx
    k1 = torch.zeros(1, L, 2)                         # at least one row: the C ABI takes no null banks
    k2 = torch.zeros(1, L, 2)
    k1[0, :n], k2[0, :n] = torch.as_tensor(p1), torch.as_tensor(p2)
    Ed = torch.as_tensor(np.asarray(E, dtype=np.float64).reshape(1, 3, 3)).to(dev)
    R, t, _, _, cnt, _, _, m, X = recover_pose_device(
        k1.to(dev), k2.to(dev), Ed, rows.to(dev), torch.zeros(1, L, device=dev),
        torch.tensor([int(idx.numel())], dtype=torch.int32, device=dev), cam, distance_thresh=distance_thresh,
        refine_iters=refine_iters, want_mask=True, want_points=True)
    k = idx.numpy()
    out_mask = np.zeros((n, 1), dtype=np.uint8)
    out_mask[k, 0] = m[0, :k.size].cpu().numpy()
    pts = np.zeros((4, n))
    pts[3] = 1.0
    pts[:3, k] = X[0, :k.size].cpu().numpy().astype(np.float64).T
    return int(cnt[0]), R[0].cpu().numpy(), t[0].cpu().numpy().reshape(3, 1), out_mask, pts


def solve_pnp_device(points, kpts, pairs, scores, counts, camera, pair_index=None, threshold=3.0, iters=1024,
                     seed=0, refine_iters=10, want_mask=False, workspace=None):
    """Camera pose per 2D-3D match list on device: points (F1,N,3) fp32 (NaN where a keypoint has no
    point), keypoints (F2,M,2) fp32 pixels of the camera ``camera`` ((fx, fy, cx, cy) or a 3x3 matrix),
    padded lists pairing point i with keypoint j -> ops.ransac_pnp's (R (P,3,3), t (P,3), pairs, scores,
    counts, rms (P,2)[, mask]) on device, x_cam ~ R X + t in the points' units.  A list without a model
    (fewer than 4 usable rows, or only degenerate samples) has R, t all zeros and an empty list."""
    fx, fy, cx, cy = _intrinsics(camera)
    return ops.ransac_pnp(points, kpts, pairs, scores, counts, fx, fy, cx, cy, pair_index=pair_index,
                          threshold=threshold, iters=iters, seed=seed, refine_iters=refine_iters,
                          want_mask=want_mask, workspace=workspace)


def triangulate_device(kpts1, kpts2, pairs, scores, counts, R, t, camera, pair_index=None, threshold=3.0,
                       min_parallax_deg=1.0, distance_thresh=50.0, refine_iters=10, want_mask=False):
    """The 3-D point of every row of the lists under a known relative pose per list (x2 ~ R x1 + t, R (P,3,3),
    t (P,3), e.g. solve_pnp_device's), in the units of t: midpoint of the rays, then refine_iters
    Levenberg-Marquardt trials on the pixel error in both views.  A row is kept iff its rays are not parallel,
    its point lies in front of both cameras closer than distance_thresh, the angle between its two rays is at
    least min_parallax_deg and its reprojection error is below threshold px in both views.  camera: (fx, fy,
    cx, cy) or a 3x3 matrix, shared by both images.  -> ops.triangulate's (points (P,L,3) fp32 in the
    camera-1 frame, zero where not kept, kept pairs, scores, counts[, mask (P,L)]) on device.  A list whose
    R is all zero (no model) or not finite keeps no row."""
    fx, fy, cx, cy = _intrinsics(camera)
    return ops.triangulate(kpts1, kpts2, pairs, scores, counts, R, t, fx, fy, cx, cy, pair_index=pair_index,
                           threshold=threshold, max_parallax_cos=math.cos(math.radians(min_parallax_deg)),
                           distance_thresh=distance_thresh, refine_iters=refine_iters, want_mask=want_mask)


def _log_so3(R):
    """Rotation matrix -> axis-angle vector (3,) (NumPy; the angle in [0, pi])."""
    c = np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0)
    th = float(np.arccos(c))
    w = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    if th < 1e-7:
        return 0.5 * w
    if np.pi - th < 1e-5:                             # near pi: the axis from the symmetric part
        k = int(np.argmax(np.diag(R)))
        a = R[:, k] + np.eye(3)[k]
        a = a / np.linalg.norm(a)
        if w @ a < 0.0:
            a = -a
        return th * a
    return th / (2.0 * np.sin(th)) * w


def solve_pnp_ransac(object_points, image_points, camera_matrix, dist_coeffs=None, iterations_count=1024,
                     reprojection_error=3.0, seed=0, refine_iters=10):
    """cv2.solvePnPRansac(objectPoints, imagePoints, K, distCoeffs, iterationsCount=, reprojectionError=,
    flags=SOLVEPNP_P3P) on the device: (n,3) points, (n,2) pixels -> (retval, rvec (3,1), tvec (3,1),
    inliers (k,1) int32 or None), x_cam ~ R(rvec) X + tvec.  A row is an inlier when its squared
    reprojection error is < reprojection_error^2 (cv2: <=) and it lies in front of the camera (cv2 does not
    test depth).  There is no distortion model: non-zero dist_coeffs raise ValueError.  n < 4 or no model
    gives (False, zeros, zeros, None).  n <= 16384."""
    if not torch.cuda.is_available():
        raise RuntimeError("sslam_b200 needs a CUDA device (no CPU fallback)")
    if dist_coeffs is not None and np.any(np.asarray(dist_coeffs, dtype=np.float64) != 0.0):
        raise ValueError("solve_pnp_ransac: lens distortion is not modelled; undistort the points first")
    cam = _intrinsics(camera_matrix)
    X = np.ascontiguousarray(np.asarray(object_points, dtype=np.float32).reshape(-1, 3))
    uv = np.ascontiguousarray(np.asarray(image_points, dtype=np.float32).reshape(-1, 2))
    if X.shape[0] != uv.shape[0]:
        raise ValueError("solve_pnp_ransac: object_points and image_points must hold the same number of points")
    n = X.shape[0]
    zeros = np.zeros((3, 1))
    if n < 4:
        return False, zeros, zeros.copy(), None
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = torch.arange(n, dtype=torch.int32).reshape(1, n, 1).expand(1, n, 2).contiguous()
    R, t, _, _, cnt, _, mask = solve_pnp_device(
        torch.as_tensor(X).reshape(1, n, 3).to(dev), torch.as_tensor(uv).reshape(1, n, 2).to(dev), rows.to(dev),
        torch.zeros(1, n, device=dev), torch.tensor([n], dtype=torch.int32, device=dev), cam,
        threshold=reprojection_error, iters=iterations_count, seed=seed, refine_iters=refine_iters, want_mask=True)
    R, t = R[0].cpu().numpy(), t[0].cpu().numpy()
    if not R.any():
        return False, zeros, zeros.copy(), None
    inl = np.flatnonzero(mask[0].cpu().numpy()).astype(np.int32).reshape(-1, 1)
    return True, _log_so3(R).reshape(3, 1), t.reshape(3, 1), inl


def _first_row(pairs, counts, mask, K):
    """The lowest row k < counts[p] with mask[p, k] set and 0 <= j = pairs[p, k, 1] < K of each keypoint j of
    list p, by a scatter-min of row indices (deterministic) -> (P, K) int64, L where there is none."""
    P, L = pairs.shape[0], pairs.shape[1]
    dev = pairs.device
    k = torch.arange(L, device=dev)
    j = pairs[..., 1].to(torch.int64)
    keep = (k[None] < counts.to(torch.int64)[:, None]) & mask.to(torch.bool) & (j >= 0) & (j < K)
    col = torch.where(keep, j, torch.full_like(j, K))             # dropped rows go to a spare column
    first = torch.full((P, K + 1), L, dtype=torch.int64, device=dev)
    first.scatter_reduce_(1, col, k[None].expand(P, L), reduce="amin", include_self=True)
    return first[:, :K]


def point_map(pairs, counts, points, mask, num_keypoints, R=None, t=None, into=None):
    """Carry one step's 3-D points to the keypoints of the next: for list p, every row k < counts[p] with
    mask[p, k] set and 0 <= j = pairs[p, k, 1] < num_keypoints gives map[p, j] = R[p] points[p, k] + t[p]
    (points[p, k] without R, t).  A keypoint in several such rows takes the lowest row (a scatter-min of row
    indices: deterministic).  -> (P, num_keypoints, 3) fp32 on device, NaN where a keypoint has no point.
    With ``into`` (P, num_keypoints, 3), its finite entries are kept and the rows fill only the others.
    pairs (P,L,2), counts (P,), points (P,L,3) and mask (P,L) index the same rows — for recover_pose_device,
    its input lists with want_mask / want_points; for solve_pnp_device, its input lists with its mask and
    its (R, t); for triangulate_device, its input lists with its mask and points and the (R, t) it was given.
    Device-only, no synchronisation, capturable in a CUDA graph."""
    P, L = pairs.shape[0], pairs.shape[1]
    K = int(num_keypoints)
    dev = pairs.device
    first = _first_row(pairs, counts, mask, K)
    has = first < L
    if L == 0:
        out = torch.full((P, K, 3), float("nan"), dtype=torch.float32, device=dev)
    else:
        X = points.to(torch.float64).gather(1, first.clamp(max=L - 1)[..., None].expand(P, K, 3))
        if R is not None:
            X = torch.einsum("pij,pkj->pki", R.to(torch.float64).reshape(P, 3, 3), X) + \
                t.to(torch.float64).reshape(P, 1, 3)
        out = torch.where(has[..., None], X, torch.full_like(X, float("nan"))).to(torch.float32)
    if into is None:
        return out
    into = into.to(torch.float32)
    return torch.where(torch.isfinite(into).all(-1, keepdim=True), into, out)


def rows_with_points(pairs, scores, counts, point_maps):
    """Restrict each list to its rows (i, j) whose point point_maps[p, i] is finite, in input order, so that
    solve_pnp_device spends no sample on a row without a point.  pairs (P,L,2), scores (P,L), counts (P,),
    point_maps (P,N,3) -> (pairs (P,L,2) int32 -1 padded, scores (P,L) fp32 0 padded, counts (P,) int32) on
    device.  No synchronisation, capturable."""
    P, L = pairs.shape[0], pairs.shape[1]
    N = point_maps.shape[1]
    dev = pairs.device
    k = torch.arange(L, device=dev)
    i = pairs[..., 0].to(torch.int64)
    keep = (k[None] < counts.to(torch.int64)[:, None]) & (i >= 0) & (i < N)
    if N:
        X = point_maps.gather(1, i.clamp(0, N - 1)[..., None].expand(P, L, 3))
        keep &= torch.isfinite(X).all(-1)
    pos = torch.where(keep, keep.to(torch.int64).cumsum(1) - 1, torch.full_like(i, L))   # dropped: spare column
    rows = torch.full((P, L + 1, 2), -1, dtype=torch.int32, device=dev)
    rows.scatter_(1, pos[..., None].expand(P, L, 2), pairs.to(torch.int32))
    sc = torch.zeros(P, L + 1, dtype=torch.float32, device=dev)
    sc.scatter_(1, pos, scores.to(torch.float32))
    return rows[:, :L].contiguous(), sc[:, :L].contiguous(), keep.sum(1).to(torch.int32)


def track_and_map(point_maps, kpts_a, kpts_b, pairs, scores, counts, camera, pair_index, threshold=3.0, iters=1024,
                  seed=0, refine_iters=10, min_parallax_deg=1.0, distance_thresh=50.0, tri_refine_iters=10,
                  want_links=False):
    """One batched step of sequence tracking with map growth.  List p pairs keypoints i of frame a with
    keypoints j of frame b, (a, b) = pair_index[p] into the banks kpts_a (Fa,Ka,2) and kpts_b (Fb,Kb,2);
    point_maps (P,Ka,3) holds the 3-D point of each keypoint of list p's frame a (NaN where there is none).

      1. rows_with_points, then solve_pnp_device: the pose (R, t) of frame b in the map's units;
      2. the PnP inliers' points are carried onto frame b's keypoints with (R, t) (point_map);
      3. every row of the input lists is triangulated under (R, t) (triangulate_device);
      4. the new points fill the keypoints of frame b that have no carried point (point_map(into=...)).

    threshold (px) is the PnP's inlier threshold and the triangulation's reprojection gate; iters, seed and
    refine_iters go to the PnP, min_parallax_deg, distance_thresh and tri_refine_iters to the triangulation.
    -> (R (P,3,3), t (P,3), PnP pairs, scores, counts, next point maps (P,Kb,3) fp32) on device.  A list
    without a PnP model has R, t all zeros and an all-NaN next map.  No synchronisation, capturable in a CUDA
    graph.

    With ``want_links`` also (link (P,Kb) int32, born (P,Kb) bool), the provenance window_tracks chains into
    multi-frame tracks: for each keypoint j of frame b with a point, link[j] is the keypoint i of frame a of
    the row that gave j its point — the lowest PnP-inlier row with that j when the point was carried (born
    0), the lowest kept triangulation row with that j when it was triangulated (born 1); -1 and 0 where j
    has no point."""
    maps = point_maps.to(torch.float32).contiguous()
    P, Kb = pairs.shape[0], kpts_b.shape[1]
    dev = pairs.device
    rows, sc, n = rows_with_points(pairs, scores, counts, maps)
    idx = pair_index.to(torch.int32)
    pnp_idx = torch.stack([torch.arange(P, dtype=torch.int32, device=dev), idx[:, 1]], 1)
    R, t, pp, ps, pc, _, mask = solve_pnp_device(maps, kpts_b, rows, sc, n, camera, pair_index=pnp_idx,
                                                 threshold=threshold, iters=iters, seed=seed,
                                                 refine_iters=refine_iters, want_mask=True)
    Na = maps.shape[1]
    X = maps.gather(1, rows[..., 0].to(torch.int64).clamp(0, max(Na - 1, 0))[..., None].expand(P, -1, 3)) \
        if Na else torch.zeros(P, rows.shape[1], 3, device=dev)
    carried = point_map(rows, n, X, mask, Kb, R, t)
    pts, _, _, _, tmask = triangulate_device(kpts_a, kpts_b, pairs, scores, counts, R, t, camera, pair_index=idx,
                                             threshold=threshold, min_parallax_deg=min_parallax_deg,
                                             distance_thresh=distance_thresh, refine_iters=tri_refine_iters,
                                             want_mask=True)
    nxt = point_map(pairs, counts, pts, tmask, Kb, R, t, into=carried)
    if not want_links:
        return R, t, pp, ps, pc, nxt
    fc = _first_row(rows, n, mask, Kb)
    ft = _first_row(pairs, counts, tmask, Kb)
    L = pairs.shape[1]
    has_c, has_t = fc < L, ft < L
    ic = rows[..., 0].to(torch.int64).gather(1, fc.clamp(max=max(L - 1, 0))) if L else fc
    it = pairs[..., 0].to(torch.int64).gather(1, ft.clamp(max=max(L - 1, 0))) if L else ft
    fin = torch.isfinite(nxt).all(-1)
    link = torch.where(fin & has_c, ic, torch.where(fin & has_t, it, torch.full_like(ic, -1)))
    return R, t, pp, ps, pc, nxt, link.to(torch.int32), fin & ~has_c & has_t


def window_tracks(maps, links, born, R, t):
    """Multi-frame tracks of a window of W frames from the provenance of its W-1 tracking steps.

    maps (P,W,K,3) point map of each window frame (NaN where a keypoint has none); links, born (P,W-1,K)
    track_and_map's link / born of the step into frame w (index w-1); R (P,W,3,3), t (P,W,3) absolute poses,
    x_w ~ R_w X + t_w, in any world frame.  Every keypoint of frame 0 with a point roots a track; a keypoint
    j of frame w >= 1 with a point inherits the track of keypoint link[j] of frame w-1 when it is not born
    and that keypoint has a track, and roots a new track at (w, j) otherwise.  A born track also observes
    (w-1, link[j]) when that keypoint has no track (the lowest such j claims it).  A track observes at most
    one keypoint per frame, the lowest j.  Its point is R_w^T (M_w[j] - t_w) of its root (w, j), in double.
    -> (obs (P,N,W) int32 keypoint of track n in frame w, -1 none; points (P,N,3) fp32 world, NaN padded;
    counts (P,) int32; track_of (P,W,K) int32, -1 none), N = W*K, tracks in ascending root order (w-major,
    then j).  Device-only, no synchronisation, capturable in a CUDA graph."""
    P, W, K = maps.shape[0], maps.shape[1], maps.shape[2]
    N = W * K
    dev = maps.device
    fin = torch.isfinite(maps).all(-1)
    j = torch.arange(K, device=dev)[None].expand(P, K)
    none = torch.full((P, K), -1, dtype=torch.int64, device=dev)
    rid, claims = [torch.where(fin[:, 0], j, none)], [none]      # root (w*K + j) of each keypoint's track
    for w in range(1, W):
        lk = links[:, w - 1].to(torch.int64)
        bn = born[:, w - 1].to(torch.bool)
        ok = (lk >= 0) & (lk < K)
        lc = lk.clamp(0, K - 1)
        prev = rid[w - 1].gather(1, lc)
        inherit = fin[:, w] & ~bn & ok & (prev >= 0)
        rid.append(torch.where(inherit, prev, torch.where(fin[:, w], w * K + j, none)))
        cand = fin[:, w] & bn & ok & (prev < 0)
        first = torch.full((P, K + 1), K, dtype=torch.int64, device=dev)
        first.scatter_reduce_(1, torch.where(cand, lc, K), j, reduce="amin", include_self=True)
        claims.append(torch.where(cand & (first.gather(1, lc) == j), lk, none))
    rid = torch.stack(rid, 1).reshape(P, N)
    flat = torch.arange(N, device=dev)[None]
    is_root = rid == flat
    pos = is_root.to(torch.int64).cumsum(1) - 1
    track_of = torch.where(rid >= 0, pos.gather(1, rid.clamp(min=0)), -1).reshape(P, W, K)
    counts = is_root.sum(1).to(torch.int32)
    obs = []
    for w in range(W):
        tw = track_of[:, w]
        m = torch.full((P, N + 1), K, dtype=torch.int64, device=dev)
        m.scatter_reduce_(1, torch.where(tw >= 0, tw, N), j, reduce="amin", include_self=True)
        obs.append(torch.where(m[:, :N] < K, m[:, :N], -1))
    for w in range(1, W):                                           # born tracks claim (w-1, link)
        cl = claims[w]
        tgt = torch.full((P, N + 1), -1, dtype=torch.int64, device=dev)
        tgt.scatter_(1, torch.where(cl >= 0, track_of[:, w], N), cl)
        obs[w - 1] = torch.where(tgt[:, :N] >= 0, tgt[:, :N], obs[w - 1])
    obs = torch.stack(obs, 2).to(torch.int32)
    Rd = R.to(torch.float64).reshape(P, W, 3, 3)
    X = torch.einsum("pwji,pwkj->pwki", Rd, maps.to(torch.float64) - t.to(torch.float64).reshape(P, W, 1, 3))
    pts = torch.full((P, N + 1, 3), float("nan"), dtype=torch.float32, device=dev)
    pts.scatter_(1, torch.where(is_root, pos, N)[..., None].expand(P, N, 3), X.reshape(P, N, 3).to(torch.float32))
    return obs.contiguous(), pts[:, :N].contiguous(), counts, track_of.to(torch.int32).contiguous()


def window_map(track_of, points, R, t, obs=None, mask=None):
    """The point maps (P,W,K,3) fp32 of the window frames from the tracks' points (P,N,3) (usually refined by
    bundle_adjust_device): M_w[j] = R_w X + t_w in double for the track of (w, j) (window_tracks' track_of),
    NaN where there is none.  With bundle_adjust_device's ``mask`` (P,N,W) and the ``obs`` it was given, a
    keypoint that is an observation of a track with at least two observations and whose mask entry is 0
    (an outlier, or not used) gets NaN; tracks of a single observation cannot be judged and keep their
    points.  The newest frame's slice feeds the next track_and_map.  Device-only, capturable."""
    P, W, K = track_of.shape
    N = points.shape[1]
    dev = track_of.device
    tr = track_of.to(torch.int64)
    keep = tr >= 0
    X = points.to(torch.float64).gather(1, tr.clamp(0, max(N - 1, 0)).reshape(P, W * K, 1).expand(P, W * K, 3))
    M = torch.einsum("pwij,pwkj->pwki", R.to(torch.float64).reshape(P, W, 3, 3), X.reshape(P, W, K, 3)) + \
        t.to(torch.float64).reshape(P, W, 1, 3)
    if mask is not None:
        ob = obs.to(torch.int64)
        seen = ob >= 0
        bad = seen & (mask == 0) & (seen.sum(2, keepdim=True) >= 2)
        drop = torch.zeros(P, W, K + 1, dtype=torch.bool, device=dev)
        drop.scatter_(2, torch.where(bad, ob, K).permute(0, 2, 1), True)
        keep = keep & ~drop[..., :K]
    return torch.where(keep[..., None], M, torch.full_like(M, float("nan"))).to(torch.float32)


def bundle_adjust_device(kpts, frame_index, obs, points, counts, R, t, camera, fixed=2, huber=3.0, threshold=3.0,
                         refine_iters=10, want_mask=False):
    """Sliding-window bundle adjustment (csrc/bundle_adjust.cu) of P windows: the poses of the last W - fixed
    frames and the tracks' points refined jointly on the pixel error of every observation, Huber-robust at
    ``huber`` px (inf: least squares), by Levenberg-Marquardt on the Schur complement.  kpts (F,K,2) pixel
    bank, frame_index (P,W) its slots, obs / points / counts as window_tracks returns them, R (P,W,3,3), t
    (P,W,3) absolute poses; camera (fx, fy, cx, cy) or a 3x3 matrix.  The default fixed = 2 pins the
    monocular scale.  -> ops.bundle_adjust's (R, t, points, rms (P,2), accepted (P,)[, mask (P,N,W)]) on
    device."""
    fx, fy, cx, cy = _intrinsics(camera)
    return ops.bundle_adjust(kpts, frame_index, obs, points, counts, R, t, fx, fy, cx, cy, fixed=fixed, huber=huber,
                             threshold=threshold, refine_iters=refine_iters, want_mask=want_mask)
