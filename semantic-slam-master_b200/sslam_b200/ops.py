"""Tensor-in / tensor-out wrappers over the C ABI.  All tensors live on the current CUDA device;
work is enqueued on torch's current stream; nothing here synchronises."""

import ctypes

import torch

from . import _lib

SIM_F32, SIM_TF32X3, SIM_BF16, SIM_F16X3 = 0, 1, 2, 3
M1, M2, M3, M4, M5 = 1, 2, 3, 4, 5


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("sslam_b200 operates on CUDA tensors only (no CPU fallback)")


def launch_count():
    return int(_lib.load().sslam_launch_count())


def profile_enable(on=True):
    """Bracket every library kernel launch with CUDA events (benchmarks only)."""
    _lib.check(_lib.load().sslam_profile_enable(1 if on else 0))


def profile_read():
    """{kernel kind: (total ms, launches)} for the launches recorded since profile_enable()."""
    lib = _lib.load()
    out = {}
    for k in range(lib.sslam_profile_kinds()):
        ms, n = ctypes.c_double(0), ctypes.c_uint64(0)
        _lib.check(lib.sslam_profile_read(k, ctypes.byref(ms), ctypes.byref(n)))
        if n.value:
            out[lib.sslam_profile_kind_name(k).decode()] = (ms.value, int(n.value))
    return out


class Workspace:
    """Grow-only device scratch buffer (one per stream of use)."""

    def __init__(self):
        self.buf = None

    def get(self, nbytes, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        return self.buf


_default_ws = {}


def _ws(kind, nbytes, device):
    key = (kind, device.index, torch.cuda.current_stream().cuda_stream)
    w = _default_ws.setdefault(key, Workspace())
    return w.get(nbytes, device)


def decode_topk(saliency, num_keypoints, nms_radius=2, min_score_percentile=0.5, floor=0.1,
                from_logits=False, out=None, workspace=None):
    """Fused decode of B maps: saliency (B,H,W) or (B,H,W,1) fp32 ->
    keypoints (B,K,2) fp32 (x,y), scores (B,K) fp32, info (B,4) int32."""
    lib = _lib.load()
    _need_cuda(saliency)
    sal = saliency[..., 0] if saliency.dim() == 4 else saliency
    if sal.dtype != torch.float32:
        raise RuntimeError("decode_topk expects fp32 saliency")
    sal = sal.contiguous()
    B, H, W = sal.shape
    K = int(num_keypoints)
    if out is None:
        kp = torch.empty(B, K, 2, dtype=torch.float32, device=sal.device)
        sc = torch.empty(B, K, dtype=torch.float32, device=sal.device)
        info = torch.empty(B, 4, dtype=torch.int32, device=sal.device)
    else:
        kp, sc, info = out
    need = lib.sslam_decode_workspace_bytes(B, H, W, K)
    ws = workspace if workspace is not None else _ws("decode", need, sal.device)
    _lib.check(lib.sslam_decode_topk_f32(_ptr(sal), int(bool(from_logits)), B, H, W, K,
                                         int(nms_radius), float(min_score_percentile), float(floor),
                                         _ptr(kp), _ptr(sc), _ptr(info), _ptr(ws), ws.numel(),
                                         _stream()))
    return kp, sc, info


def nms(saliency, radius):
    """saliency (B,H,W) fp32 -> same shape, non-maxima zeroed."""
    lib = _lib.load()
    _need_cuda(saliency)
    sal = saliency.contiguous()
    B, H, W = sal.shape
    out = torch.empty_like(sal)
    _lib.check(lib.sslam_nms_f32(_ptr(sal), B, H, W, int(radius), _ptr(out), _stream()))
    return out


def gather_bilinear(features, keypoints, pixel_coords=False, out=None, pair=False):
    """features (B,h,w,C) fp32 NHWC, keypoints (B,N,2) fp32 -> (B,N,C) fp32.
    pair=True returns instead the fp16 (hi, lo) pair consumed by refiner_forward (no fp32 copy)."""
    lib = _lib.load()
    _need_cuda(features, keypoints)
    feat = features.contiguous()
    kp = keypoints.contiguous()
    if feat.dtype != torch.float32 or kp.dtype != torch.float32:
        raise RuntimeError("gather_bilinear expects fp32 tensors")
    B, h, w, C = feat.shape
    N = kp.shape[1]
    hi = lo = None
    if pair:
        hi = torch.empty(B, N, C, dtype=torch.float16, device=feat.device)
        lo = torch.empty(B, N, C, dtype=torch.float16, device=feat.device)
    elif out is None:
        out = torch.empty(B, N, C, dtype=torch.float32, device=feat.device)
    _lib.check(lib.sslam_gather_bilinear_f32(_ptr(feat), _ptr(kp), B, h, w, C, N,
                                             1 if pixel_coords else 0, _ptr(out), _ptr(hi), _ptr(lo),
                                             _stream()))
    return (hi, lo) if pair else out


def l2norm_rows(x, eps=1e-12, out=None, out_bf16=None, want_bf16=False, pair=None):
    """x (..., D) fp32 -> x / max(||x||, eps); optionally also a bf16 copy.  `pair` = (hi, lo) fp16
    tensors of x's shape additionally receive the result as the fp16 pair hi + lo*2^-11 that
    match_top2(mode=SIM_F16X3) consumes directly."""
    lib = _lib.load()
    _need_cuda(x)
    xc = x.contiguous()
    D = xc.shape[-1]
    rows = xc.numel() // D
    if out is None:
        out = torch.empty_like(xc)
    if want_bf16 and out_bf16 is None:
        out_bf16 = torch.empty(xc.shape, dtype=torch.bfloat16, device=xc.device)
    hi, lo = _check_pair(pair, rows * D)
    _lib.check(lib.sslam_l2norm_rows(_ptr(xc), rows, D, float(eps), _ptr(out), _ptr(out_bf16), _ptr(hi),
                                     _ptr(lo), _stream()))
    return (out, out_bf16) if want_bf16 else out


def _check_pair(pair, numel):
    if pair is None:
        return None, None
    hi, lo = pair
    for t in (hi, lo):
        if t.dtype != torch.float16 or not t.is_contiguous() or t.numel() != numel:
            raise RuntimeError("fp16 pair outputs must be contiguous fp16 tensors of the result's size")
    return hi, lo


class RefinerPlan:
    """Device-side state for sslam_refiner_forward_f32: pointer table + packed fp16 hi/lo weight pairs of
    one DescriptorRefiner-shaped parameter set (state_dict order)."""

    def __init__(self, tensors, C, Hd, D, blocks):
        lib = _lib.load()
        _need_cuda(*tensors)
        self.tensors = [t.detach().contiguous() for t in tensors]
        for t in self.tensors:
            if t.dtype != torch.float32:
                raise RuntimeError("refiner parameters must be fp32")
        self.C, self.Hd, self.D, self.blocks = int(C), int(Hd), int(D), int(blocks)
        assert len(self.tensors) == 4 + 8 * self.blocks
        self.ptrs = (ctypes.c_void_p * len(self.tensors))(*[t.data_ptr() for t in self.tensors])
        dev = self.tensors[0].device
        nbytes = lib.sslam_refiner_packed_bytes(self.C, self.Hd, self.D, self.blocks)
        self.packed = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.sslam_refiner_pack_weights(self.ptrs, self.C, self.Hd, self.D, self.blocks,
                                                  _ptr(self.packed), nbytes, _stream()))


def refiner_forward(plan, x, eps=1e-12, want_bf16=False, workspace=None, out=None, out16=None, out_pair=None):
    """x (..., C) fp32 — or the (hi, lo) fp16 pair from gather_bilinear(pair=True) —
    -> unit-norm descriptors (rows, D) fp32 [and bf16 copy] [and, into out_pair = (hi, lo), the fp16
    pair the f16x3 matcher multiplies]."""
    lib = _lib.load()
    x_hi = x_lo = None
    if isinstance(x, (tuple, list)):
        x_hi, x_lo = (t.contiguous() for t in x)
        _need_cuda(x_hi, x_lo)
        if x_hi.dtype != torch.float16 or x_lo.dtype != torch.float16 or x_hi.shape[-1] != plan.C:
            raise RuntimeError("refiner_forward expects an fp16 (hi, lo) pair with %d channels" % plan.C)
        xc, rows = None, x_hi.numel() // plan.C
        ref = x_hi
    else:
        _need_cuda(x)
        xc = x.contiguous()
        if xc.dtype != torch.float32 or xc.shape[-1] != plan.C:
            raise RuntimeError("refiner_forward expects fp32 input with %d channels" % plan.C)
        rows = xc.numel() // plan.C
        ref = xc
    xc_dev = ref.device
    if out is None:
        out = torch.empty(rows, plan.D, dtype=torch.float32, device=xc_dev)
    if want_bf16 and out16 is None:
        out16 = torch.empty(rows, plan.D, dtype=torch.bfloat16, device=xc_dev)
    for t in (out, out16):
        if t is not None and (not t.is_contiguous() or t.numel() != rows * plan.D):
            raise RuntimeError("refiner_forward: output buffers must be contiguous (rows, D)")
    p_hi, p_lo = _check_pair(out_pair, rows * plan.D)
    need = lib.sslam_refiner_workspace_bytes(rows, plan.C, plan.Hd, plan.D, plan.blocks)
    ws = workspace if workspace is not None else _ws("refiner", need, xc_dev)
    _lib.check(lib.sslam_refiner_forward_f32(plan.ptrs, _ptr(plan.packed), _ptr(xc), _ptr(x_hi), _ptr(x_lo),
                                             rows, plan.C,
                                             plan.Hd, plan.D, plan.blocks, float(eps), _ptr(out),
                                             _ptr(out16), _ptr(p_hi), _ptr(p_lo), _ptr(ws), ws.numel(),
                                             _stream()))
    return (out, out16) if want_bf16 else out


def refiner_range_check():
    """Waits for the current stream and raises SslamError(SSLAM_ERANGE) if a refiner forward on this device
    stored an activation outside the fp16 range of the f16x3 arithmetic (|x| >= 65504, NaN or inf) since the
    last check; such descriptors must not be used (run DescriptorRefiner with mlp="torch").  Not capturable."""
    _lib.check(_lib.load().sslam_refiner_range_check(_stream()))


def match_top2(bank1, bank2, pair_index=None, mode=SIM_F16X3, num_pairs=None, workspace=None):
    """Row top-2 / column argmax of S_p = D1_p . D2_p^T without storing S.

    The default arithmetic is SIM_F16X3 — the tcgen05/TMEM tile GEMM with fp32-level accuracy (D % 8 == 0);
    SIM_F32 is the CUDA-core exact kernel kept as the explicit cross-check (and for D % 8 != 0).

    bank1 (F1,N,D), bank2 (F2,M,D); pair_index (P,2) int32 selects (a,b) per pair, default (p,p).
    With mode=SIM_F16X3 a bank may also be the (hi, lo) fp16 pair written by l2norm_rows /
    refiner_forward (both banks then), which skips the split pass.
    Returns dict(nn12, best12, second12 (P,N); nn21, best21 (P,M))."""
    lib = _lib.load()
    presplit = isinstance(bank1, (tuple, list))
    if presplit != isinstance(bank2, (tuple, list)):
        raise RuntimeError("either both descriptor banks are fp16 (hi, lo) pairs or neither")
    if presplit:
        if mode != SIM_F16X3:
            raise RuntimeError("fp16 (hi, lo) descriptor banks are the operand format of SIM_F16X3 only")
        (bank1, bank1_lo), (bank2, bank2_lo) = bank1, bank2
        _need_cuda(bank1, bank1_lo, bank2, bank2_lo)
        for t in (bank1, bank1_lo, bank2, bank2_lo):
            if t.dtype != torch.float16 or not t.is_contiguous():
                raise RuntimeError("fp16 (hi, lo) descriptor banks must be contiguous fp16")
        if bank1.shape != bank1_lo.shape or bank2.shape != bank2_lo.shape:
            raise RuntimeError("hi and lo halves of a descriptor bank must have the same shape")
    else:
        bank1_lo = bank2_lo = None
        _need_cuda(bank1, bank2, pair_index)
        if not (bank1.is_contiguous() and bank2.is_contiguous()):
            raise RuntimeError("descriptor banks must be contiguous")
        want = torch.bfloat16 if mode == SIM_BF16 else torch.float32
        if bank1.dtype != want or bank2.dtype != want:
            raise RuntimeError(f"mode {mode} expects {want} descriptor banks")
    N, D = bank1.shape[-2], bank1.shape[-1]
    M = bank2.shape[-2]
    if pair_index is not None:
        pair_index = pair_index.to(torch.int32).contiguous()
        P = pair_index.shape[0]
    else:
        P = int(num_pairs) if num_pairs is not None else min(bank1.shape[0], bank2.shape[0])
    dev = bank1.device
    res = dict(nn12=torch.empty(P, N, dtype=torch.int32, device=dev),
               best12=torch.empty(P, N, dtype=torch.float32, device=dev),
               second12=torch.empty(P, N, dtype=torch.float32, device=dev),
               nn21=torch.empty(P, M, dtype=torch.int32, device=dev),
               best21=torch.empty(P, M, dtype=torch.float32, device=dev))
    F1 = bank1.numel() // (N * D)
    F2 = bank2.numel() // (M * D)
    need = lib.sslam_match_workspace_bytes(F1, F2, P, N, M, D, mode)
    ws = workspace if workspace is not None else _ws("match", need, dev)
    _lib.check(lib.sslam_match_top2(_ptr(bank1), _ptr(bank1_lo), F1, _ptr(bank2), _ptr(bank2_lo), F2,
                                    _ptr(pair_index), int(mode), P, N, M,
                                    D, _ptr(res["nn12"]), _ptr(res["best12"]), _ptr(res["second12"]),
                                    _ptr(res["nn21"]), _ptr(res["best21"]), _ptr(ws), ws.numel(),
                                    _stream()))
    return res


def match_finalize(variant, top, params, pair_index=None, scores1=None, scores2=None,
                   inten1=None, inten2=None):
    """Apply acceptance rule `variant` to the output of match_top2.
    Returns pairs (P,N,2) int32 (-1 padded), pair_scores (P,N) fp32, counts (P,) int32."""
    lib = _lib.load()
    nn12 = top["nn12"]
    P, N = nn12.shape
    M = top["nn21"].shape[1]
    dev = nn12.device
    if pair_index is not None:
        pair_index = pair_index.to(torch.int32).contiguous()
    pairs = torch.empty(P, N, 2, dtype=torch.int32, device=dev)
    pscores = torch.empty(P, N, dtype=torch.float32, device=dev)
    counts = torch.empty(P, dtype=torch.int32, device=dev)
    prm = (ctypes.c_double * 8)(*([float(v) for v in params] + [0.0] * (8 - len(params))))
    for t in (scores1, scores2, inten1, inten2):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("score / intensity banks must be contiguous fp32")
    _lib.check(lib.sslam_match_finalize(int(variant), prm, _ptr(pair_index), P, N, M, _ptr(nn12),
                                        _ptr(top["best12"]), _ptr(top["second12"]), _ptr(top["nn21"]),
                                        _ptr(top["best21"]), _ptr(scores1), _ptr(scores2),
                                        _ptr(inten1), _ptr(inten2), _ptr(pairs), _ptr(pscores),
                                        _ptr(counts), _stream()))
    return pairs, pscores, counts


# ---------------------------------------------------------------------------------- evaluation (N4)
def nn_points(kpts1, kpts2, H=None, pair_index=None, num_pairs=None):
    """Nearest keypoint of set 2 for every (optionally homography-warped) keypoint of set 1.

    kpts1 (F1,N,2), kpts2 (F2,M,2) fp32; H (P,3,3) float64 or None; pair_index (P,2) int32 or None.
    Returns (min_dist (P,N) float64 with H / float32 without, argmin (P,N) int32)."""
    lib = _lib.load()
    _need_cuda(kpts1, kpts2, H, pair_index)
    k1, k2 = kpts1.contiguous(), kpts2.contiguous()
    if k1.dtype != torch.float32 or k2.dtype != torch.float32:
        raise RuntimeError("nn_points expects fp32 keypoints")
    F1, N = k1.shape[0], k1.shape[1]
    F2, M = k2.shape[0], k2.shape[1]
    if pair_index is not None:
        pair_index = pair_index.to(torch.int32).contiguous()
        P = pair_index.shape[0]
    else:
        P = int(num_pairs) if num_pairs is not None else min(F1, F2)
    if H is not None:
        H = H.to(torch.float64).contiguous()
        if H.numel() != P * 9:
            raise RuntimeError("nn_points: H must hold one 3x3 matrix per pair")
    md = torch.empty(P, N, dtype=torch.float64 if H is not None else torch.float32, device=k1.device)
    am = torch.empty(P, N, dtype=torch.int32, device=k1.device)
    _lib.check(lib.sslam_nn_points(_ptr(k1), F1, _ptr(k2), F2, _ptr(H), _ptr(pair_index), P, N, M, _ptr(md),
                                   _ptr(am), _stream()))
    return md, am


def gt_matches(min_dist, argmin, threshold=3.0, want_pairs=True):
    """Rows with min_dist < threshold as (i, argmin[i]), ascending i.
    Returns pairs (P,N,2) int32 -1-padded (or None), counts (P,) int32."""
    lib = _lib.load()
    _need_cuda(min_dist, argmin)
    P, N = min_dist.shape
    md = min_dist.contiguous()
    pairs = torch.empty(P, N, 2, dtype=torch.int32, device=md.device) if want_pairs else None
    counts = torch.empty(P, dtype=torch.int32, device=md.device)
    _lib.check(lib.sslam_gt_matches(_ptr(md), _ptr(argmin.contiguous()), int(md.dtype == torch.float64),
                                    float(threshold), P, N, _ptr(pairs), _ptr(counts), _stream()))
    return pairs, counts


def eval_matches(pred_pairs, pred_counts, gt_pairs, gt_counts, num_kpts1):
    """tp / fp / fn per pair (P,3) int32 of predicted against ground-truth padded pair lists."""
    lib = _lib.load()
    _need_cuda(pred_pairs, pred_counts, gt_pairs, gt_counts)
    P = pred_pairs.shape[0]
    pp, gp = pred_pairs.to(torch.int32).contiguous(), gt_pairs.to(torch.int32).contiguous()
    scratch = torch.empty(P, int(num_kpts1), dtype=torch.int32, device=pp.device)
    out = torch.empty(P, 3, dtype=torch.int32, device=pp.device)
    _lib.check(lib.sslam_eval_matches(_ptr(pp), _ptr(pred_counts.to(torch.int32).contiguous()), pp.shape[1],
                                      _ptr(gp), _ptr(gt_counts.to(torch.int32).contiguous()), gp.shape[1], P,
                                      int(num_kpts1), _ptr(scratch), _ptr(out), _stream()))
    return out


# ---------------------------------------------------------------------------------- geometric verification
def ransac_homography(kpts1, kpts2, pairs, pair_scores, counts, pair_index=None, num_pairs=None, threshold=3.0,
                      iters=1024, seed=0, want_mask=False, workspace=None):
    """RANSAC homography per padded match list (sslam_ransac_homography).

    kpts1 (F1,N,2), kpts2 (F2,M,2) fp32; pairs (P,L,2) int32, pair_scores (P,L) fp32, counts (P,) int32 as
    match_finalize returns them; pair_index (P,2) int32 selects (a,b) per pair, default (p,p).
    Returns (H (P,3,3) float64, h33 = 1, all zeros where there is no model; inlier pairs (P,L,2) int32 in
    input order, -1 padded; their scores (P,L); counts (P,) int32[; inlier mask (P,L) uint8 per input row])."""
    return _ransac("homography", kpts1, kpts2, pairs, pair_scores, counts, pair_index, num_pairs, threshold, iters,
                   seed, want_mask, workspace)


def ransac_fundamental(kpts1, kpts2, pairs, pair_scores, counts, pair_index=None, num_pairs=None, threshold=3.0,
                       iters=1024, seed=0, want_mask=False, workspace=None):
    """RANSAC fundamental matrix per padded match list (sslam_ransac_fundamental): 7-point samples,
    symmetric epipolar error, 8-point refit.  Arguments as for ransac_homography; ``iters`` counts samples.
    Returns (F (P,3,3) float64 with x2^T F x1 = 0, unit Frobenius norm, all zeros where there is no model;
    inlier pairs, scores, counts[, inlier mask]) in ransac_homography's format."""
    return _ransac("fundamental", kpts1, kpts2, pairs, pair_scores, counts, pair_index, num_pairs, threshold,
                   iters, seed, want_mask, workspace)


_RANSAC_SYMBOLS = {"homography": ("sslam_ransac_homography", "sslam_ransac_workspace_bytes", 1),
                   "fundamental": ("sslam_ransac_fundamental", "sslam_ransac_fundamental_workspace_bytes", 3)}


def ransac_workspace_bytes(P, L, iters, model="homography"):
    """Workspace bytes ransac_homography / ransac_fundamental need for P lists of stride L."""
    return getattr(_lib.load(), _RANSAC_SYMBOLS[model][1])(int(P), int(L), int(iters))


def _ransac(model, kpts1, kpts2, pairs, pair_scores, counts, pair_index, num_pairs, threshold, iters, seed,
            want_mask, workspace):
    name = "ransac_" + model
    lib = _lib.load()
    _need_cuda(kpts1, kpts2, pairs, pair_scores, counts, pair_index)
    k1, k2 = kpts1.contiguous(), kpts2.contiguous()
    if k1.dtype != torch.float32 or k2.dtype != torch.float32:
        raise RuntimeError(f"{name} expects fp32 keypoints")
    pr = pairs.to(torch.int32).contiguous()
    ps = pair_scores.to(torch.float32).contiguous()
    cn = counts.to(torch.int32).contiguous()
    F1, N = k1.shape[0], k1.shape[1]
    F2, M = k2.shape[0], k2.shape[1]
    P, L = pr.shape[0], pr.shape[1]
    if pair_index is not None:
        pair_index = pair_index.to(torch.int32).contiguous()
        if pair_index.shape[0] != P:
            raise RuntimeError(f"{name}: pair_index must hold one (a, b) row per match list")
    elif num_pairs is not None and int(num_pairs) != P:
        raise RuntimeError(f"{name}: num_pairs differs from the number of match lists")
    dev = pr.device
    G = torch.empty(P, 3, 3, dtype=torch.float64, device=dev)
    out_pairs = torch.empty(P, L, 2, dtype=torch.int32, device=dev)
    out_scores = torch.empty(P, L, dtype=torch.float32, device=dev)
    out_counts = torch.empty(P, dtype=torch.int32, device=dev)
    mask = torch.empty(P, L, dtype=torch.uint8, device=dev) if want_mask else None
    fn, ws_fn, _ = _RANSAC_SYMBOLS[model]
    need = getattr(lib, ws_fn)(P, L, int(iters))
    ws = workspace if workspace is not None else _ws("ransac", need, dev)
    _lib.check(getattr(lib, fn)(_ptr(k1), F1, _ptr(k2), F2, _ptr(pair_index), P, N, M, _ptr(pr),
                                _ptr(ps), _ptr(cn), L, int(iters), float(threshold),
                                int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(G), _ptr(out_pairs),
                                _ptr(out_scores), _ptr(out_counts), _ptr(mask), _ptr(ws), ws.numel(),
                                _stream()))
    return (G, out_pairs, out_scores, out_counts) + ((mask,) if want_mask else ())


def ransac_workspace_views(workspace, P, L, iters, model="homography"):
    """Views of what sslam_ransac_homography (model="homography") or sslam_ransac_fundamental
    (model="fundamental") leaves at the start of its workspace: per-slot inlier counts (P,S) int32 (-1
    degenerate), S = iters for the homography and 3*iters for the fundamental matrix (slots 3s..3s+2
    belong to sample s); the best slot (P,) int32 (-1 none); and the best slot's inlier mask before the
    refit (P,L) uint8."""
    def up(x):
        return (x + 255) // 256 * 256
    S = iters * _RANSAC_SYMBOLS[model][2]
    o_best = up(P * S * 4)
    o_mask = o_best + up(P * 4)
    w = workspace
    return (w[:P * S * 4].view(torch.int32).reshape(P, S),
            w[o_best:o_best + P * 4].view(torch.int32),
            w[o_mask:o_mask + P * L].reshape(P, L))


# ---------------------------------------------------------------------------------- optional decode front stage (J1)
def heatmap_from_cells(logits, cell=8, border=0):
    """(B, cell*cell+1, Hc, Wc) fp32 cell logits -> (B, Hc*cell, Wc*cell) heatmap: channel softmax,
    dustbin dropped, depth-to-space, border mask.  Off-by-default decode mode (no reference code)."""
    lib = _lib.load()
    _need_cuda(logits)
    x = logits.contiguous()
    if x.dtype != torch.float32 or x.dim() != 4 or x.shape[1] != cell * cell + 1:
        raise RuntimeError("heatmap_from_cells expects fp32 (B, cell*cell+1, Hc, Wc) logits")
    B, _, Hc, Wc = x.shape
    heat = torch.empty(B, Hc * cell, Wc * cell, dtype=torch.float32, device=x.device)
    _lib.check(lib.sslam_heatmap_from_cells_f32(_ptr(x), B, Hc, Wc, int(cell), int(border), _ptr(heat), _stream()))
    return heat


# ---------------------------------------------------------------------------------- selector head (N2)
class SelectorPlan:
    """Packed fp16 (hi, lo) weights of the selector's 3x3 convolution, reordered to [hidden][tap][C]."""

    def __init__(self, conv1_weight, conv1_bias, conv2_weight, conv2_bias):
        lib = _lib.load()
        _need_cuda(conv1_weight, conv1_bias, conv2_weight, conv2_bias)
        w1 = conv1_weight.detach().contiguous()
        if w1.dtype != torch.float32 or w1.dim() != 4 or tuple(w1.shape[2:]) != (3, 3):
            raise RuntimeError("selector head expects an fp32 [hidden, C, 3, 3] convolution weight")
        self.hidden, self.C = int(w1.shape[0]), int(w1.shape[1])
        self.b1 = conv1_bias.detach().contiguous()
        self.w2 = conv2_weight.detach().reshape(-1).contiguous()
        self.b2 = conv2_bias.detach().reshape(-1).contiguous()
        if self.w2.numel() != self.hidden or self.b2.numel() != 1:
            raise RuntimeError("selector head expects a [1, hidden, 1, 1] second convolution")
        nbytes = lib.sslam_selector_packed_bytes(self.C, self.hidden)
        self.packed = torch.empty(nbytes, dtype=torch.uint8, device=w1.device)
        _lib.check(lib.sslam_selector_pack_weights(_ptr(w1), self.C, self.hidden, _ptr(self.packed), nbytes,
                                                   _stream()))


def selector_head(plan, features, apply_sigmoid=True, out=None, workspace=None):
    """features (B,H,W,C) fp32 NHWC -> (B,H,W) fp32 saliency (or logits): 3x3 conv + ReLU + 1x1 conv
    [+ sigmoid] as one tcgen05 implicit-GEMM kernel."""
    lib = _lib.load()
    _need_cuda(features)
    f = features.contiguous()
    if f.dtype != torch.float32 or f.dim() != 4 or f.shape[-1] != plan.C:
        raise RuntimeError("selector_head expects fp32 (B,H,W,%d) features" % plan.C)
    B, H, W, C = f.shape
    if out is None:
        out = torch.empty(B, H, W, dtype=torch.float32, device=f.device)
    need = lib.sslam_selector_workspace_bytes(B, H, W, C)
    ws = workspace if workspace is not None else _ws("selector", need, f.device)
    _lib.check(lib.sslam_selector_head_f32(_ptr(f), _ptr(plan.packed), _ptr(plan.b1), _ptr(plan.w2), _ptr(plan.b2),
                                           B, H, W, C, plan.hidden, 1 if apply_sigmoid else 0, _ptr(out), _ptr(ws),
                                           ws.numel(), _stream()))
    return out
