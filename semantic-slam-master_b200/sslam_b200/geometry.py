"""Geometric verification of match lists on the device (csrc/ransac.cu): RANSAC homography, for planar
scenes and rotating cameras, and RANSAC fundamental matrix (the epipolar constraint), for a camera that
translates through a 3-D scene.

Device API — ``verify_homography_device`` / ``verify_fundamental_device`` take banks of keypoint sets and
the padded lists the matcher produced (``pairs [P,N,2]``, ``pair_scores [P,N]``, ``counts [P]``) and
return, still on the device, one model per pair plus the inlier rows in the same padded format, so every
consumer of match lists (``evaluation.to_match_lists``, ``write_match_lists``,
``pack_match_records``, ``dist.gather_match_lists``) takes the verified lists unchanged and the
estimated ``H`` feeds ``evaluation.ground_truth_matches_device`` directly.

Host API — ``find_homography`` has the arguments and the return shape of ``cv2.findHomography(src,
dst, cv2.RANSAC, thresh)``: ``(H (3,3) float64 or None, mask (n,1) uint8)``; ``find_fundamental`` those
of ``cv2.findFundamentalMat(pts1, pts2, cv2.FM_RANSAC, thresh)``.
"""

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
