"""Seeded synthetic inputs shaped like the reference's data (SURVEY.md §8(d)).

There is no TUM RGB-D data, no DINOv3 checkpoint and no network, so every benchmark and parity
test feeds the hot path the tensors it would see *after* the backbone and the selector head:
a saliency map (B, H, W, 1) fp32 and an NHWC feature map (B, H/16, W/16, 384) fp32.  A sequence
is a crop window sliding over a fixed "world canvas" (TUM fr1/desk-like small motion: one patch
every 8 frames), so consecutive frames overlap and mutual matches exist.

All randomness comes from ``torch.Generator`` objects with the seeds listed in SURVEY.md §8(d);
identical tensors are handed to the oracle and to the kernels.  The keypoint-level two-view banks at the
end (``two_view_bank``, ``two_view_lists``), for epipolar geometry, are drawn with NumPy generators.
"""

import numpy as np
import torch
import torch.nn.functional as F

PATCH = 16
MARGIN = 600
FEAT_DIM = 384


class WorldCanvas:
    """Smoothed-noise logits canvas + iid feature canvas for one synthetic sequence."""

    def __init__(self, seq_id=0, height=480, width=640, feat_dim=FEAT_DIM, device="cpu"):
        assert height % PATCH == 0 and width % PATCH == 0
        self.seq_id, self.H, self.W, self.C = int(seq_id), int(height), int(width), int(feat_dim)
        self.device = torch.device(device)
        g = torch.Generator(device="cpu").manual_seed(1000 + self.seq_id)
        ch, cw = self.H + 2 * MARGIN, self.W + 2 * MARGIN
        raw = torch.randn(ch, cw, generator=g)
        smooth = F.avg_pool2d(raw[None, None], kernel_size=5, stride=1, padding=2,
                              count_include_pad=False)[0, 0]
        self.logits = (smooth * 4.0).to(self.device)
        self.feats = torch.randn(ch // PATCH, cw // PATCH, self.C, generator=g).to(self.device)

    def frame(self, t):
        """Return (logits (H, W), features (H/16, W/16, C)) of frame ``t`` on ``self.device``."""
        ox = (PATCH * (t // 8)) % (2 * MARGIN)
        oy = 0
        gen_dev = "cuda" if self.device.type == "cuda" else "cpu"
        g = torch.Generator(device=gen_dev).manual_seed(2000 + int(t) + 100003 * self.seq_id)
        lg = self.logits[oy:oy + self.H, ox:ox + self.W]
        lg = lg + 0.05 * torch.randn(self.H, self.W, generator=g, device=self.device)
        h, w = self.H // PATCH, self.W // PATCH
        ft = self.feats[oy // PATCH:oy // PATCH + h, ox // PATCH:ox // PATCH + w]
        ft = ft + 0.02 * torch.randn(h, w, self.C, generator=g, device=self.device)
        return lg.contiguous(), ft.contiguous()


def make_sequence(num_frames, seq_id=0, height=480, width=640, feat_dim=FEAT_DIM,
                  device="cpu", start=0, stride=1, out_saliency=None, out_features=None):
    """Frames ``start, start+stride, ...`` of sequence ``seq_id``.

    Returns saliency (T, H, W, 1) fp32 — ``torch.sigmoid`` of the logits, computed once on
    ``device`` and shared by every implementation — and features (T, H/16, W/16, C) fp32 NHWC.
    Pre-allocated (e.g. pinned) outputs may be supplied.
    """
    canvas = WorldCanvas(seq_id, height, width, feat_dim, device)
    h, w = height // PATCH, width // PATCH
    sal = out_saliency if out_saliency is not None else torch.empty(
        num_frames, height, width, 1, device=canvas.device)
    feat = out_features if out_features is not None else torch.empty(
        num_frames, h, w, feat_dim, device=canvas.device)
    for i in range(num_frames):
        lg, ft = canvas.frame(start + i * stride)
        sal[i, :, :, 0].copy_(torch.sigmoid(lg))
        feat[i].copy_(ft)
    return sal, feat


def make_pairs(num_pairs, height=480, width=640, feat_dim=FEAT_DIM, device="cpu"):
    """c3-style independent pairs: frames (2p, 2p+1) of sequences p = 0..num_pairs-1.
    Returns saliency (P, 2, H, W, 1) and features (P, 2, h, w, C)."""
    sals, feats = [], []
    for p in range(num_pairs):
        s, f = make_sequence(2, seq_id=p, height=height, width=width, feat_dim=feat_dim,
                             device=device, start=2 * p)
        sals.append(s)
        feats.append(f)
    return torch.stack(sals, 0), torch.stack(feats, 0)


def native_grid_case(batch=4, grid=28, feat_dim=FEAT_DIM, seed=7):
    """c0: the reference-native 28x28 patch grid — iid features; the saliency comes from the
    selector head with ``torch.manual_seed(0)`` weights (made by the caller)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(batch, grid, grid, feat_dim, generator=g)


def noisy_permutation_descriptors(n, d=256, noise=0.05, seed=0, m=None):
    """Unit-norm descriptor sets (n, d) and (m, d) where set 2 is a noisy permutation of set 1
    (plus fresh rows if m > n); used by matcher tests."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    m = n if m is None else m
    a = F.normalize(torch.randn(n, d, generator=g), dim=-1)
    perm = torch.randperm(n, generator=g)
    b = a[perm][:min(n, m)] + noise * torch.randn(min(n, m), d, generator=g)
    if m > n:
        b = torch.cat([b, torch.randn(m - n, d, generator=g)], 0)
    b = F.normalize(b, dim=-1)
    return a.contiguous(), b.contiguous(), perm


def _rotation(w):
    """Rodrigues: axis-angle vector (3,) -> rotation matrix (3,3)."""
    th = float(np.linalg.norm(w))
    if th == 0.0:
        return np.eye(3)
    k = np.asarray(w, dtype=np.float64) / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1.0 - np.cos(th)) * (Kx @ Kx)


def two_view_bank(num_sets=2, num_points=2048, seed=0, noise=0.0, baseline=(0.2, 0.4), direction=None,
                  focal=525.0, height=480, width=640):
    """Keypoint banks of one static 3-D scene seen by a moving pinhole camera (general motion, so the
    epipolar geometry is identifiable — unlike make_sequence, whose frames are translated crops of a flat
    canvas).  Point k is drawn at a uniform pixel of set 0 and a depth of 4-10 m; each later camera pose
    moves by a small random rotation (0.02-0.05 rad) and a translation of ``baseline`` (m, uniform) in a
    random direction, or along ``direction`` (3,) when given (a sideways motion keeps the epipoles far
    outside the image, where the epipolar lines constrain every point).
    Keypoint k of every set is the projection of point k (plus ``noise`` px Gaussian), rounded to fp32.

    Returns (bank (num_sets, num_points, 2) float32 ndarray in the [F,K,2] layout, F (num_sets-1, 3, 3)
    float64): F[s] is the true fundamental matrix of sets (s, s+1), x_{s+1}^T F x_s = 0, at unit Frobenius
    norm with its largest-|entry| element positive."""
    rng = np.random.default_rng(seed)
    K = np.array([[focal, 0.0, (width - 1) / 2.0], [0.0, focal, (height - 1) / 2.0], [0.0, 0.0, 1.0]])
    Ki = np.linalg.inv(K)
    pix = rng.uniform([0.0, 0.0], [width - 1.0, height - 1.0], size=(num_points, 2))
    X = (np.concatenate([pix, np.ones((num_points, 1))], 1) @ Ki.T) * rng.uniform(4.0, 10.0, (num_points, 1))
    bank = np.empty((num_sets, num_points, 2))
    Fs = np.empty((max(num_sets - 1, 0), 3, 3))
    for s in range(num_sets):
        if s:
            axis = rng.normal(size=3)
            R = _rotation(axis / np.linalg.norm(axis) * rng.uniform(0.02, 0.05))
            t = rng.normal(size=3) if direction is None else np.asarray(direction, dtype=np.float64).copy()
            t *= rng.uniform(*baseline) / np.linalg.norm(t)
            X = X @ R.T + t
            tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
            Fm = Ki.T @ tx @ R @ Ki
            Fm /= np.linalg.norm(Fm)
            Fs[s - 1] = -Fm if Fm.reshape(9)[np.abs(Fm).argmax()] < 0 else Fm
        p = X @ K.T
        bank[s] = p[:, :2] / p[:, 2:3] + (rng.normal(0.0, noise, (num_points, 2)) if noise > 0 else 0.0)
    return bank.astype(np.float32), Fs


def two_view_lists(counts, list_stride, num_points, inlier_frac=0.7, seed=1):
    """Padded match lists over two_view_bank sets: list p holds counts[p] rows (i, j) with ascending
    distinct i; j = i (a true correspondence) with probability ``inlier_frac``, a uniform keypoint
    otherwise.  -> pairs (P, L, 2) int32 (-1 padded), scores (P, L) fp32, counts (P,) int32, true (P, L)
    bool (j = i)."""
    rng = np.random.default_rng(seed)
    P = len(counts)
    pairs = np.full((P, list_stride, 2), -1, dtype=np.int32)
    scores = np.zeros((P, list_stride), dtype=np.float32)
    true = np.zeros((P, list_stride), dtype=bool)
    for p, n in enumerate(counts):
        i = np.sort(rng.choice(num_points, size=int(n), replace=False))
        keep = rng.random(int(n)) < inlier_frac
        j = np.where(keep, i, rng.integers(0, num_points, size=int(n)))
        pairs[p, :n, 0], pairs[p, :n, 1] = i, j
        scores[p, :n] = rng.random(int(n)).astype(np.float32)
        true[p, :n] = j == i
    return pairs, scores, np.asarray(counts, dtype=np.int32), true
