/*
 * sslam_b200.h — C ABI of libsslam_b200.so, the B200 (sm_100a) replacement for the per-frame
 * learned-feature front-end of Siverteh/semantic-slam-master.
 *
 * The reference is pure Python and has no FFI of its own; its boundary for this path is the
 * method surface cited at each entry point below (paths relative to <reference>/semantic-slam/).
 * A reference-side binding (ctypes) is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (e.g. torch tensors) unless it says host;
 *  - the library never allocates caller-visible memory, never synchronises the stream and never
 *    throws across the ABI; work is enqueued on `stream` (a cudaStream_t) and the call returns;
 *  - return value: SSLAM_OK (0) or a negative SSLAM_E* code; sslam_last_error() gives the text
 *    (thread-local);
 *  - there is no CPU fallback: on a machine without an sm_100 device every compute entry point
 *    returns SSLAM_ENODEVICE.
 *  - one process may drive several devices: device properties, kernel attributes and occupancy
 *    answers are cached per device; calls act on the calling thread's current device.
 *  - tie rules: top-k order is (score descending, linear index y*W+x ascending); argmax returns
 *    the lowest maximal index (NumPy / torch-CPU behaviour).
 */
#ifndef SSLAM_B200_H_
#define SSLAM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSLAM_ABI_VERSION 4

enum {
  SSLAM_OK = 0,
  SSLAM_EINVAL = -1,       /* bad argument (null pointer, negative size, floor < 0 ...)        */
  SSLAM_EUNSUPPORTED = -2, /* shape outside what the kernels implement (see each entry point)  */
  SSLAM_EWORKSPACE = -3,   /* workspace smaller than sslam_*_workspace_bytes()                 */
  SSLAM_ECUDA = -4,        /* a CUDA runtime call failed; text in sslam_last_error()           */
  SSLAM_ENODEVICE = -5,    /* no CUDA device of compute capability 10.x                        */
  SSLAM_ERANGE = -6        /* an activation left the fp16 range of the f16x3 arithmetic        */
};

/* decode `info` columns, int32 [B,4] */
enum {
  SSLAM_INFO_BRANCH = 0,     /* 0 main (keypoint_selector.py:120-128), 1 lower percentile (:139-156),
                                2 raw padding (:157-173), 3 raw top-k (:174-184),
                                -1 the reference would raise: topk with k > H*W (:166,178)      */
  SSLAM_INFO_NCAND = 1,      /* candidates above the main threshold; -1 when the fast path proved
                                "at least K" without computing the exact count                  */
  SSLAM_INFO_TIES = 2,       /* entries equal to the k-th score that were left out               */
  SSLAM_INFO_NLOCALMAX = 3   /* NMS survivors above the lowest floor                             */
};

/* similarity arithmetic for sslam_match_top2 */
enum {
  SSLAM_SIM_F32 = 0,    /* fp32 FMA on CUDA cores (exact-mode reference implementation)          */
  SSLAM_SIM_TF32X3 = 1, /* tcgen05 kind::tf32, 3-term hi/lo split, fp32 accumulate in TMEM       */
  SSLAM_SIM_BF16 = 2,   /* tcgen05 kind::f16 on bf16 copies, fp32 accumulate in TMEM             */
  SSLAM_SIM_F16X3 = 3   /* fp32 in/out; x = hi + lo*2^-11 with hi, lo fp16 (22 mantissa bits), three
                           kind::f16 MMAs (hi.hi, hi.lo, lo.hi) at the full 16-bit tensor rate, fp32
                           accumulate in TMEM; same accuracy class as TF32X3 at half the tensor time
                           and half the operand bytes.  Requires |x| < 65504.                   */
};

/* acceptance rule for sslam_match_finalize; params[] meaning per variant */
enum {
  SSLAM_MATCH_M1 = 1, /* visualize_matches.py:102-124      params[0] = ratio_thresh, params[1] = 0:
                         compare `sim > second*ratio` in fp32 (NumPy >= 2 scalar promotion, the
                         behaviour the golden fixtures were written under), 1: in double (NumPy < 2,
                         which the reference's requirements.txt:1 pins)                           */
  SSLAM_MATCH_M2 = 2, /* visualize_matches_sequence.py:106-197  params = {saliency_weight,
                         min_saliency, min_descriptor_sim, min_intensity, 1 - saliency_weight
                         (rounded to fp32 by the caller, as Python computes it in double)}       */
  SSLAM_MATCH_M3 = 3, /* test/test_descriptor_quality.py:97-142  params[0] = ratio_threshold     */
  SSLAM_MATCH_M4 = 4, /* train.py:410-449                  mutual NN only                        */
  SSLAM_MATCH_M5 = 5  /* test/test_tracking.py:159-161     params[0] = match_threshold, no mutual */
};

int sslam_abi_version(void);

/* Copies the calling thread's last error text into buf (host); returns its length. */
int sslam_last_error(char* buf, size_t len);

/* 0 when the current CUDA device is compute capability 10.x, else SSLAM_ENODEVICE / SSLAM_ECUDA. */
int sslam_device_check(void);

/* Number of kernel launches (not memsets) this process enqueued through the library so far. */
uint64_t sslam_launch_count(void);

/* Optional per-kernel timing for benchmarks: while enabled, every kernel launch of the library is
 * bracketed by CUDA events on its launch stream.  sslam_profile_enable() also clears the records;
 * sslam_profile_read() waits for the recorded events of one kernel kind (0 .. kinds-1) and returns
 * their summed duration and count.  Off by default (no events, no overhead). */
int sslam_profile_enable(int on);
int sslam_profile_kinds(void);
const char* sslam_profile_kind_name(int kind);
int sslam_profile_read(int kind, double* total_ms, uint64_t* launches);

/* ---------------------------------------------------------------------------------------------
 * Heatmap decode.  Replaces KeypointSelector.select_keypoints / _apply_nms and, with
 * from_logits != 0, the sigmoid tail of KeypointSelector.forward
 * (models/keypoint_selector.py:69-207, 209-226, 61-62).
 *
 *   sal      [B,H,W] fp32 saliency (or logits)        kpts_xy [B,K,2] fp32 (x,y), integer valued
 *   scores   [B,K] fp32                               info    [B,4] int32 (SSLAM_INFO_*), may be NULL
 *   pct      min_score_percentile (reference default 0.50);  floor: 0.1 in the reference (>= 0)
 *   nms_radius 0..8
 * Limits: 1 <= K <= 16384, H*W <= 2^24 (torch.quantile's own limit).
 * All B maps are decoded by the same launches; there is no host synchronisation.
 */
size_t sslam_decode_workspace_bytes(int B, int H, int W, int K);
int sslam_decode_topk_f32(const float* sal, int from_logits, int B, int H, int W, int K,
                          int nms_radius, float pct, float floor, float* kpts_xy, float* scores,
                          int32_t* info, void* ws, size_t ws_bytes, void* stream);

/* NMS only (KeypointSelector._apply_nms, keypoint_selector.py:209-226): out = sal where sal equals
 * its (2r+1)^2 neighbourhood maximum, else 0.  sal/out [B,H,W]. */
int sslam_nms_f32(const float* sal, int B, int H, int W, int nms_radius, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Bilinear descriptor sampling.  Replaces DinoBackbone.extract_at_keypoints
 * (models/dino_backbone.py:114-152) with ATen-identical coordinate arithmetic and zero padding.
 *   feat [B,h,w,C] fp32 NHWC      kpts [B,N,2] fp32 (x,y)      out [B,N,C] fp32
 *   coords: 0 = keypoints are in patch units (drop-in);
 *           1 = keypoints are in pixel units and DinoBackbone.pixel_to_patch (:167-178,
 *               (p-8)/16) is applied first.
 *   out may be NULL when the fp16 pair (out_hi, out_lo: [B,N,C] fp16 each, value = hi + lo*2^-11,
 *   the operand format of sslam_refiner_forward_f32) is requested instead of / in addition to fp32.
 */
int sslam_gather_bilinear_f32(const float* feat, const float* kpts, int B, int h, int w, int C,
                              int N, int coords, float* out, void* out_hi, void* out_lo,
                              void* stream);

/* Row-wise L2 normalisation, the tail of DescriptorRefiner.forward
 * (models/descriptor_refiner.py:86): out = in / max(||in||_2, eps).
 *   in [rows,D] fp32;  out_f32 [rows,D] fp32 or NULL;  out_bf16 [rows,D] bf16 or NULL;
 *   out_hi / out_lo [rows,D] fp16 or both NULL: the normalised value as the fp16 pair
 *   hi + lo*2^-11 that sslam_match_top2(SSLAM_SIM_F16X3) multiplies (saves its own split pass). */
int sslam_l2norm_rows(const float* in, int rows, int D, float eps, float* out_f32,
                      void* out_bf16, void* out_hi, void* out_lo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * DescriptorRefiner forward (models/descriptor_refiner.py:58-91, 108-126): Linear+ReLU, `blocks`
 * pre-LayerNorm residual blocks, Linear, L2 normalise — tcgen05 f16x3 GEMMs (fp32-level accuracy)
 * with fused bias / residual / ReLU epilogues.
 *   params : HOST array of 4 + 8*blocks DEVICE pointers (fp32), in state_dict order:
 *            input_proj.{weight [Hd,C], bias}; per block norm1.{weight,bias}, fc1.{weight [Hd,Hd],
 *            bias}, norm2.{weight,bias}, fc2.{weight,bias}; output_proj.{weight [D,Hd], bias}
 *   packed : device buffer of sslam_refiner_packed_bytes(), filled once per weight set by
 *            sslam_refiner_pack_weights() (fp16 hi/lo pairs of the Linear weights, LayerNorms folded)
 *   x [rows,C] fp32 (or NULL with the pair x_hi/x_lo [rows,C] fp16 from sslam_gather_bilinear_f32)
 *   -> out_f32 [rows,D] fp32 and/or out_bf16 [rows,D] bf16 and/or the fp16 pair out_hi/out_lo
 *      [rows,D] (see sslam_l2norm_rows), unit L2 norm
 * Arithmetic: fp16 hi/lo pairs (22 significant bits), three kind::f16 MMAs per product, fp32
 * accumulation; |activation| must stay below 65504.  C, Hd multiples of 8, D of 4; Hd <= 1024;
 * LayerNorm eps is torch's default 1e-5.
 */
size_t sslam_refiner_packed_bytes(int C, int Hd, int D, int blocks);
int sslam_refiner_pack_weights(const float* const* params, int C, int Hd, int D, int blocks,
                               void* packed, size_t packed_bytes, void* stream);
size_t sslam_refiner_workspace_bytes(int rows, int C, int Hd, int D, int blocks);
int sslam_refiner_forward_f32(const float* const* params, const void* packed, const float* x,
                              const void* x_hi, const void* x_lo,
                              int rows, int C, int Hd, int D, int blocks, float eps_norm,
                              float* out_f32, void* out_bf16, void* out_hi, void* out_lo,
                              void* ws, size_t ws_bytes, void* stream);
/* Range guard of the fp16-pair arithmetic.  Every GEMM epilogue of sslam_refiner_forward_f32 watches the
 * activations it stores: when the sum of squares of 64 consecutive columns of a row reaches 65504^2 (so at
 * the latest when one |activation| >= 65504, where the fp16 hi part becomes inf), or is NaN / inf (which
 * is also how an out-of-range INPUT shows up), a sticky flag is set on the device.  This call waits for
 * `stream`, returns SSLAM_ERANGE if the flag was set by any forward on the current device since the last
 * call (and clears it), SSLAM_OK otherwise.  The descriptors of a flagged forward are not to be used:
 * run the fp32 PyTorch body (DescriptorRefiner(mlp="torch")) for such weights / inputs. */
int sslam_refiner_range_check(void* stream);

/* ---------------------------------------------------------------------------------------------
 * Matching primitive shared by M1..M5: over the virtual S_p = D1_p . D2_p^T (never stored)
 *   per row    nn12 (lowest argmax), best12, second12 (second entry of the row sorted descending,
 *              -inf when M == 1);     [P,N]
 *   per column nn21 (lowest argmax), best21;   [P,M]
 * bank1 holds F1 descriptor sets [F1,N,D], bank2 holds F2 sets [F2,M,D] (the banks may alias, e.g.
 * bank2 = bank1 + N*D for consecutive-frame matching).  Pair p reads set a of bank1 and set b of
 * bank2 where (a,b) = pair_index[p] if pair_index != NULL (int32 [P,2], device) else (p,p).  `dtype` is SSLAM_SIM_*; banks are fp32 for
 * SSLAM_SIM_F32 / TF32X3 / F16X3 and bf16 for SSLAM_SIM_BF16.  D % 4 == 0 (8 for bf16/f16x3), D <= 256.
 * SSLAM_SIM_F16X3 only: when bank1_lo and bank2_lo are non-NULL the banks are already split —
 * bank1 / bank2 are the fp16 hi arrays and bank1_lo / bank2_lo the fp16 lo arrays written by
 * sslam_l2norm_rows / sslam_refiner_forward_f32 — and no split pass runs.
 * Replaces visualize_matches.py:105-109,117-119; visualize_matches_sequence.py:144-146;
 * test/test_descriptor_quality.py:116-130; train.py:422-424; test/test_tracking.py:159-160.
 */
size_t sslam_match_workspace_bytes(int F1, int F2, int P, int N, int M, int D, int dtype);
int sslam_match_top2(const void* bank1, const void* bank1_lo, int F1, const void* bank2,
                     const void* bank2_lo, int F2, const int32_t* pair_index, int dtype,
                     int P, int N, int M, int D, int32_t* nn12, float* best12, float* second12,
                     int32_t* nn21, float* best21, void* ws, size_t ws_bytes, void* stream);

/* Acceptance rules + ordered compaction (ascending i).
 *   pairs [P,N,2] int32, rows beyond counts[p] are -1;  pair_scores [P,N] fp32;  counts [P] int32
 *   pair_scores: M1/M4/M5 similarity, M2 quality, M3 1 - similarity.
 *   scores1/scores2 (saliency per keypoint, banks [*,N] / [*,M]) are required for M2;
 *   inten1/inten2 optional (M2).  They are indexed by the same (a,b) as the descriptor banks.
 */
int sslam_match_finalize(int variant, const double* params /* host, 8 doubles; rounded to fp32
                         where the reference compares in fp32 */,
                         const int32_t* pair_index, int P, int N, int M, const int32_t* nn12,
                         const float* best12, const float* second12, const int32_t* nn21,
                         const float* best21, const float* scores1, const float* scores2,
                         const float* inten1, const float* inten2, int32_t* pairs,
                         float* pair_scores, int32_t* counts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Evaluation adaptors (SURVEY.md §8(f) N4) — nearest (warped) keypoint, ground-truth match lists and
 * match scoring for P keypoint-set pairs at once.  Replaces the N x M distance matrices of
 * DescriptorQualityTester.compute_ground_truth_matches / evaluate_matches
 * (test/test_descriptor_quality.py:144-183, 185-231) and RepeatabilityTester.compute_repeatability
 * (test/test_repeatability.py:79-128).
 *   kpts1 [F1,N,2], kpts2 [F2,M,2] fp32 (x,y); pair p reads sets (a,b) = pair_index[p] (int32 [P,2]) or (p,p)
 *   H     [P,9] double, row-major homographies frame1 -> frame2, or NULL
 *   min_dist [P,N]: DOUBLE when H != NULL (the reference promotes to float64 when it warps), FLOAT when
 *             H == NULL (test_repeatability.py:104-105 subtracts and norms the float32 arrays)
 *   argmin   [P,N] int32, lowest index of the minimum
 */
int sslam_nn_points(const float* kpts1, int F1, const float* kpts2, int F2, const double* H,
                    const int32_t* pair_index, int P, int N, int M, void* min_dist, int32_t* argmin,
                    void* stream);

/* rows with min_dist < threshold, ascending i, as (i, argmin[i]) (test_descriptor_quality.py:173-181);
 * pairs [P,N,2] int32 (-1 padded) may be NULL when only counts [P] (the repeatable count,
 * test_repeatability.py:116) are wanted. */
int sslam_gt_matches(const void* min_dist, const int32_t* argmin, int is_double, double threshold, int P,
                     int N, int32_t* pairs, int32_t* counts, void* stream);

/* tp / fp / fn of predicted against ground-truth lists (test_descriptor_quality.py:202-215); both
 * lists hold each first index at most once.  pred [P,pred_stride,2], gt [P,gt_stride,2] int32 with
 * their counts [P]; scratch [P,N] int32; out [P,3] int32. */
int sslam_eval_matches(const int32_t* pred, const int32_t* pred_counts, int pred_stride,
                       const int32_t* gt, const int32_t* gt_counts, int gt_stride, int P, int N,
                       int32_t* scratch, int32_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Geometric verification: RANSAC homography over the padded match lists of P pairs at once, in a
 * fixed number of launches without host synchronisation (capturable in a CUDA graph).
 *   kpts1 [F1,N,2], kpts2 [F2,M,2] fp32 (x,y); pair p reads sets (a,b) = pair_index[p] (int32 [P,2]) or
 *   (p,p), as sslam_match_top2 / sslam_nn_points do.  pairs [P,L,2] int32 rows (i,j), pair_scores [P,L],
 *   counts [P]: the output format of sslam_match_finalize (L = its N); rows k < min(counts[p], L) are used.
 *   Hypothesis h (0 <= h < iters) of a pair with n rows solves the normalised 4-point DLT (double) on 4
 *   distinct rows drawn by splitmix64: draw c (< 32, repeats redrawn) is output h*32 + c of the stream
 *   seeded with `seed`, row = (u >> 32) * n >> 32.  Samples depend on (seed, h, n) only, so a pair gives
 *   the same result alone or anywhere in a batch.  A sample is degenerate when a pivot of the 8x8 solve or
 *   h33 is below 1e-8 in magnitude (collinear or repeated points), or when its 4 draws are not distinct.
 *   Row k is an inlier of H iff ||pi(H.(x1,y1,1)) - (x2,y2)||^2 < threshold^2 (forward transfer error,
 *   strict), in fp32 with u/w and v/w formed as u*(1/w), v*(1/w).
 *   The best hypothesis has the most inliers; ties go to the lowest h.  It is refit by least squares
 *   (normalised DLT over its inliers, smallest eigenvector of the 9x9 normal matrix, double, fixed-order
 *   reductions) and the refit is kept iff it has at least as many inliers.
 *   Outputs: H [P,9] double row-major frame1 -> frame2 scaled to h33 = 1 (may be NULL); the inlier rows in
 *   input order (ascending i is preserved) as out_pairs [P,L,2] int32 (-1 padded), out_scores [P,L] (the
 *   rows' pair_scores, 0 padded), out_counts [P]; inlier_mask [P,L] uint8 per input row (may be NULL).
 *   No model — n < 4 or every hypothesis degenerate — is data: out_counts[p] = 0, H[p] all zeros, SSLAM_OK.
 *   On return the workspace starts with the inlier count of every hypothesis, int32 [P,iters] (-1:
 *   degenerate), followed at the next 256-byte boundary by the best hypothesis per pair, int32 [P] (-1:
 *   none), and at the next by the best hypothesis's inlier mask before the refit, uint8 [P,L].
 * Limits: L <= 16384, 1 <= iters <= 65536, threshold > 0.  Out-of-range keypoint indices in a row make
 * that row an outlier (and a sample containing it degenerate).
 */
size_t sslam_ransac_workspace_bytes(int P, int L, int iters);
int sslam_ransac_homography(const float* kpts1, int F1, const float* kpts2, int F2,
                            const int32_t* pair_index, int P, int N, int M,
                            const int32_t* pairs, const float* pair_scores, const int32_t* counts, int L,
                            int iters, double threshold, uint64_t seed,
                            double* H, int32_t* out_pairs, float* out_scores,
                            int32_t* out_counts, uint8_t* inlier_mask,
                            void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Epipolar verification: RANSAC fundamental matrix over the padded match lists of P pairs at once.
 * The parameters, the launches, the determinism, the outputs' format, the no-model convention and the
 * limits are those of sslam_ransac_homography; only the model differs.
 *   Sample s (0 <= s < iters; iters counts samples, as cv2's maxIters does) draws 7 distinct rows with
 *   the same sampler (draw c < 32 is output s*32 + c, repeats redrawn).  The 7-point solve runs in double
 *   with correctly rounded operations only: each image's points are normalised (centroid, sqrt(2) / mean
 *   distance); the 7x9 system of rows [u x, u y, u, v x, v y, v, x, y, 1] (x1 = (x,y), x2 = (u,v)) is
 *   reduced by Gaussian elimination with full pivoting (largest |entry| of the remaining submatrix,
 *   lowest (row, column) on ties); the two columns that never pivot, in ascending order, give the null
 *   vectors f1, f2.  The real roots of det(F2 + lam (F1 - F2)) = c3 lam^3 + c2 lam^2 + c1 lam + c0 are
 *   taken as lam in [-1, 1] from that cubic, then as mu = 1/lam in (-1, 1) from c0 mu^3 + c1 mu^2 + c2 mu
 *   + c3 (mu = 0 is F1 - F2); each interval is split at the real critical points and every bracket
 *   with a sign change is bisected 64 times.  Each root's F is denormalised (T2^T F T1), scaled to unit
 *   Frobenius norm and signed so that its largest-|entry| element (lowest index on ties) is positive.
 *   Sample s owns hypothesis slots 3s, 3s+1, 3s+2, filled in root order (the first cubic's roots
 *   ascending, then the second's); unused slots are degenerate.  A sample is degenerate when n < 7, the
 *   sampler finds no 7 distinct rows in 32 draws, the 7 points coincide in either image, a pivot is below
 *   1e-8 in magnitude (7 correspondences related by one homography give a rank-6 system, so an exactly
 *   planar or purely rotating sample is degenerate) or no root is real.
 *   Row k is an inlier of F iff both squared point-to-epipolar-line distances (cv2's FM_RANSAC error) are
 *   < threshold^2, in fp32 with the fp32 hypothesis: a2 = (F0 x1 + F1 y1) + F2, b2 = (F3 x1 + F4 y1) + F5,
 *   c2 = (F6 x1 + F7 y1) + F8, d2 = (x2 a2 + y2 b2) + c2, e2 = d2 d2 * (1 / (a2 a2 + b2 b2)); e1 likewise
 *   with F^T and the points' roles swapped.  An undefined line (NaN) makes the row an outlier.
 *   The best slot has the most inliers (lowest slot on ties).  With at least 8 inliers it is refit by the
 *   normalised 8-point least squares over them (smallest eigenvector of the 9x9 normal matrix, rank 2
 *   enforced as F' = Fn - (Fn v3) v3^T with v3 the smallest eigenvector of Fn^T Fn), kept iff it has at
 *   least as many inliers.
 *   Outputs: F [P,9] double row-major with x2^T F x1 = 0, unit Frobenius norm (may be NULL); out_pairs,
 *   out_scores, out_counts and inlier_mask as for the homography.  No model is data: F[p] all zeros, an
 *   empty list, SSLAM_OK.  On return the workspace starts with the inlier count of every slot, int32
 *   [P,3*iters] (-1: degenerate), then at the next 256-byte boundary the best slot per pair, int32 [P]
 *   (-1: none), then the best slot's inlier mask before the refit, uint8 [P,L].
 * Limits: L <= 16384, 1 <= iters <= 65536, threshold > 0.  The workspace holds 40 bytes per slot, so
 * 32 640 pairs (all pairs of 256 keyframes) at 1024 samples need about 4.0 GB.
 */
size_t sslam_ransac_fundamental_workspace_bytes(int P, int L, int iters);
int sslam_ransac_fundamental(const float* kpts1, int F1, const float* kpts2, int F2,
                             const int32_t* pair_index, int P, int N, int M,
                             const int32_t* pairs, const float* pair_scores, const int32_t* counts, int L,
                             int iters, double threshold, uint64_t seed,
                             double* F, int32_t* out_pairs, float* out_scores,
                             int32_t* out_counts, uint8_t* inlier_mask,
                             void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optional cell-softmax front stage of the decode (north_star "softmax/depth-to-space ... border
 * mask"; OFF by default — the reference code has no such mode, keypoint_selector.py:61-62 is a
 * sigmoid; the vocabulary is papers/pdfs/SuperPoint_DeTone.md:49-58):
 *   logits [B, cell*cell+1, Hc, Wc] fp32 -> softmax over channels, last channel dropped,
 *   depth-to-space to heat [B, Hc*cell, Wc*cell], pixels closer than `border` to an edge zeroed.
 * cell in {2,4,8}.  The heatmap is then decoded by sslam_decode_topk_f32.
 */
int sslam_heatmap_from_cells_f32(const float* logits, int B, int Hc, int Wc, int cell, int border,
                                 float* heat, void* stream);

/* ---------------------------------------------------------------------------------------------
 * KeypointSelector head (models/keypoint_selector.py:30-34, 56-65): Conv2d(C, hidden, 3, padding=1)
 * -> ReLU -> Conv2d(hidden, 1, 1) [-> sigmoid] on the NHWC patch-feature map, as one tcgen05
 * implicit-GEMM kernel (f16x3: fp32-level accuracy) whose epilogue contracts the hidden activations
 * with the 1x1 convolution; writes one value per pixel (SURVEY.md §8(f) N2).
 *   feat [B,H,W,C] fp32 NHWC;  packed = sslam_selector_pack_weights(conv.0.weight [hidden,C,3,3]);
 *   conv1_bias [hidden], conv2_weight [hidden] (= conv.2.weight [1,hidden,1,1]), conv2_bias [1]: fp32
 *   out [B,H,W] fp32: logits (apply_sigmoid = 0) or saliency (1).
 * C % 64 == 0, hidden % 8 == 0, hidden <= 512.
 */
size_t sslam_selector_packed_bytes(int C, int hidden);
int sslam_selector_pack_weights(const float* conv1_weight, int C, int hidden, void* packed,
                                size_t packed_bytes, void* stream);
size_t sslam_selector_workspace_bytes(int B, int H, int W, int C);
int sslam_selector_head_f32(const float* feat, const void* packed, const float* conv1_bias,
                            const float* conv2_weight, const float* conv2_bias, int B, int H, int W,
                            int C, int hidden, int apply_sigmoid, float* out, void* ws,
                            size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSLAM_B200_H_ */
