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
 * Relative pose from verified match lists: the camera motion (R, t) of each of P pairs and the
 * triangulated points, in one launch (one CTA per pair), without workspace or host synchronisation
 * (capturable in a CUDA graph), without atomics; a pair's result does not depend on its position in the
 * batch.  The banks, pair_index and the padded lists are those of sslam_ransac_fundamental (typically its
 * out_pairs / out_scores / out_counts); rows k < min(counts[p], L) are used.  E [P,9] double row-major is
 * the essential matrix of each pair (K^T F K); one pinhole camera K = [[fx,0,cx],[0,fy,cy],[0,0,1]] is
 * shared by both images of every pair.  A row is usable when its keypoint indices are in range and its
 * coordinates finite; any other row is never good and stays out of the refinement.
 *   Decomposition (double): E / |E|_F; the eigenvectors of E^T E by cyclic Jacobi, ordered by descending
 *   eigenvalue (lowest index on ties), v3 negated when det V < 0; u1 = normalise(E v1), u2 =
 *   normalise(E v2 - (u1.E v2) u1), u3 = u1 x u2; with W = [[0,1,0],[-1,0,0],[0,0,1]] (cv2's),
 *   R_a = U W V^T, R_b = U W^T V^T, t = u3; the candidates are (R_a, t), (R_b, t), (R_a, -t), (R_b, -t).
 *   Cheirality (double, correctly rounded operations): rays f1 = K^-1 x1, f2 = K^-1 x2, u = R f1;
 *   a = u.u, b = u.f2, c = f2.f2, d = u.t, e = f2.t, den = a c - b^2, z1 = (b e - c d) / den, X1 = z1 f1
 *   (camera-1 frame, |t| = 1).  A row is good iff den > 1e-12 a c, 0 < z1 < distance_thresh and
 *   0 < (R X1 + t)_z < distance_thresh (cv2.recoverPose's cheirality and distanceThresh).  The candidate
 *   with the most good rows is chosen, the lowest on ties.
 *   Refinement (refine_iters Levenberg-Marquardt trials, 0 disables it; skipped with fewer than 5 usable
 *   rows): R <- Exp(w) R (Rodrigues), t <- normalise(t + d1 b1 + d2 b2) with b1 = normalise(t x e_i),
 *   i = argmin |t_i| (lowest on ties), b2 = t x b1; residual the signed Sampson distance in pixels of every
 *   usable row, x2^T F x1 / sqrt((F x1)_0^2 + (F x1)_1^2 + (F^T x2)_0^2 + (F^T x2)_1^2), F = K^-T [t]x R K^-1
 *   (0 when the denominator is 0); analytic Jacobian dE/dw_j = [t]x [e_j]x R, dE/dd_j = [b_j]x R.  J^T J,
 *   J^T r and r^T r are reduced in fixed order once per relinearisation; lambda starts at 1e-3 times the
 *   mean of diag(J^T J); each trial solves (J^T J + lambda diag(J^T J)) x = -J^T r by Cholesky and costs
 *   the candidate; it is accepted iff the cost strictly decreases (lambda /= 10, relinearise), otherwise
 *   lambda *= 10.  The candidate's sign and branch never change.
 *   Outputs: R [P,9] and t [P,3] (unit; x2 ~ R x1 + t in camera coordinates); cand_good [P,4] the four
 *   candidates' good rows before the refinement (may be NULL); rms [P,2] the RMS Sampson distance (px)
 *   over the usable rows before and after the refinement (may be NULL); with the refined pose the
 *   cheirality is run again: pose_mask [P,L] uint8 the good rows (may be NULL), points [P,L,3] fp32 X1 of
 *   every good row and 0 elsewhere (may be NULL), and the good rows in input order as out_pairs [P,L,2]
 *   (-1 padded), out_scores [P,L] (0 padded), out_counts [P] — the matcher's list format.
 *   No pose is data: E all zeros (the fundamental RANSAC's "no model"), E not finite, sigma2 <= 1e-12
 *   sigma1, or no good row for the best candidate give R, t, rms, mask and points all zeros and an empty
 *   list, and SSLAM_OK.
 * Limits: L <= 16384, 0 <= refine_iters <= 100, distance_thresh > 0 and finite, fx, fy > 0 and finite,
 * cx, cy finite.
 */
int sslam_recover_pose(const float* kpts1, int F1, const float* kpts2, int F2, const int32_t* pair_index,
                       int P, int N, int M, const double* E, const int32_t* pairs, const float* pair_scores,
                       const int32_t* counts, int L, double fx, double fy, double cx, double cy,
                       double distance_thresh, int refine_iters,
                       double* R, double* t, int32_t* cand_good, double* rms,
                       float* points, int32_t* out_pairs, float* out_scores,
                       int32_t* out_counts, uint8_t* pose_mask, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Camera tracking: RANSAC P3P over padded 2D-3D match lists, the pose of camera 2 with respect to the
 * 3-D points of each of P lists.  Three launches for all lists, no host synchronisation (capturable in
 * a CUDA graph), no atomics; a list's result depends only on its own inputs and (iters, threshold, seed,
 * refine_iters), never on its position in the batch.
 *   points [F1,N,3] fp32 are 3-D points in some camera frame (NaN where there is no point), kpts2
 *   [F2,M,2] fp32 pixels; pair_index [P,2] selects (a, b) per list (NULL: (p, p)); pairs [P,L,2] int32,
 *   pair_scores [P,L], counts [P] as sslam_match_finalize writes them, row (i, j) pairing points[a][i]
 *   with kpts2[b][j].  Rows k < n = min(counts[p], L) are used; a row with an index out of range or a
 *   coordinate that is not finite is never an inlier and makes a sample that holds it degenerate.  One
 *   pinhole camera K = [[fx,0,cx],[0,fy,cy],[0,0,1]] for camera 2.
 *   Sample s (0 <= s < iters) draws 4 distinct rows with the sampler of sslam_ransac_homography (draw
 *   c < 32 is output s*32 + c, repeats redrawn).  Rows 0-2 go to the Lambda Twist P3P solver (Persson
 *   & Nordberg, ECCV 2018) in double with correctly rounded operations only: bearings y = normalise(
 *   (u - cx) / fx, (v - cy) / fy, 1); the cubic's root by bisection of [-B, B], B = 1 + max |k_i| (the
 *   Cauchy bound of the monic cubic), 100 steps; the rank-2 conic's eigenvectors in closed form; up to 5
 *   Gauss-Newton steps on the depths.  Among the solutions that are finite and put all four points at
 *   z > 0, row 3 picks the one with the least squared reprojection error (lowest on ties).  A sample is
 *   degenerate when n < 4, the sampler finds no 4 distinct rows, a row is not usable, the three solver
 *   points are collinear or coincident (|d12 x d13|^2 <= 1e-12 |d12|^2 |d13|^2, d1j = X1 - Xj), or no
 *   solution is real and in front of the camera.
 *   Row k is an inlier of the fp32 hypothesis (R, t) iff Zc > 0 and du^2 + dv^2 < threshold^2, in fp32
 *   without contraction: Xc = ((R0 X + R1 Y) + R2 Z) + t0 (Yc, Zc likewise), iz = 1 / Zc (correctly
 *   rounded), du = ((fx Xc) iz + cx) - u, dv = ((fy Yc) iz + cy) - v, (du du + dv dv) < t^2; a NaN is an
 *   outlier.  cv2.solvePnPRansac uses <= and no depth test.
 *   The best sample has the most inliers (lowest sample on ties).  With at least 4 inliers and
 *   refine_iters > 0 its pose is refined by Levenberg-Marquardt in 6 DOF (R <- Exp(w) R, t <- t + d) on
 *   the reprojection error in pixels of its inliers (2 residuals per row, analytic Jacobian); lambda
 *   starts at 1e-3 times the mean of diag(J^T J); each trial solves (J^T J + lambda diag(J^T J)) x =
 *   -J^T r by Cholesky and is accepted iff the cost strictly decreases (lambda /= 10), otherwise
 *   lambda *= 10.  The refined pose is kept iff it has at least as many inliers over all rows.
 *   Outputs: R [P,9] and t [P,3] double, x_cam2 ~ R X + t in the points' units; rms [P,2] the RMS
 *   reprojection error (px) over the best sample's inliers before and after the refinement (the second
 *   equals the first when the refinement is skipped or not kept; may be NULL); out_pairs, out_scores,
 *   out_counts and inlier_mask as for sslam_ransac_homography.  No model is data: R, t and rms all
 *   zeros, an empty list, SSLAM_OK; so is a best sample without any inlier.  On return the workspace starts
 *   with the inlier count of every sample, int32 [P,iters] (-1: degenerate), then at the next 256-byte
 *   boundary the best sample per list, int32 [P] (-1: none), then the best sample's inlier mask before the
 *   refinement, uint8 [P,L], then the fp32 hypotheses.
 * Limits: L <= 16384, 1 <= iters <= 65536, 0 <= refine_iters <= 100, threshold > 0 and finite, fx, fy > 0
 * and finite, cx, cy finite.  The workspace holds 52 bytes per sample, so 32 640 lists at 1024 samples
 * need about 1.7 GB.
 */
size_t sslam_ransac_pnp_workspace_bytes(int P, int L, int iters);
int sslam_ransac_pnp(const float* points, int F1, const float* kpts2, int F2, const int32_t* pair_index,
                     int P, int N, int M, const int32_t* pairs, const float* pair_scores,
                     const int32_t* counts, int L, double fx, double fy, double cx, double cy, int iters,
                     double threshold, uint64_t seed, int refine_iters,
                     double* R, double* t, double* rms, int32_t* out_pairs, float* out_scores,
                     int32_t* out_counts, uint8_t* inlier_mask, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Triangulation of match lists under a known relative pose (map growth): the 3-D point of every row of P
 * lists, x_b ~ R x_a + t, in the units of t.  One launch (one CTA per list), no workspace, no atomics, no
 * host synchronisation (capturable in a CUDA graph); a list's result does not depend on its position in
 * the batch.  The banks, pair_index and the padded lists are those of sslam_recover_pose; rows k <
 * min(counts[p], L) are used, and a row whose keypoint indices are out of range or whose coordinates are
 * not finite is never kept.  R [P,9] double row-major and t [P,3] double are each list's relative pose
 * (typically sslam_ransac_pnp's); a list whose R or t has a non-finite entry, or whose R is all zero (the
 * "no model" of every geometry entry), keeps no row.  One pinhole camera K = [[fx,0,cx],[0,fy,cy],[0,0,1]]
 * for both images.  Per row, on one thread, in double with correctly rounded operations only:
 *   Midpoint: the rays and midpoint of sslam_recover_pose's cheirality (f1 = K^-1 x1, f2 = K^-1 x2,
 *   X = z1 f1), which also gives the "rays not parallel" test den > 1e-12 a c.
 *   Refinement (refine_iters Levenberg-Marquardt trials on X, 0 keeps the midpoint): the residual is the
 *   4-vector of pixel errors pi(X) - x1, pi(R X + t) - x2 with an analytic Jacobian; lambda starts at 1e-3
 *   times the mean of diag(J^T J); each trial solves (J^T J + lambda diag(J^T J)) x = -J^T r by Cholesky,
 *   and the candidate X + x is accepted iff its depth is > 0 in both cameras and the cost strictly
 *   decreases (lambda /= 10, relinearise), otherwise lambda *= 10.
 *   Gates on the final X: the row is kept iff the rays are not parallel, 0 < z_a < distance_thresh and
 *   0 < z_b < distance_thresh, the parallax cosine X.(X - C_b) / (|X| |X - C_b|) with C_b = -R^T t is
 *   <= max_parallax_cos, and the squared reprojection error is < threshold^2 in both views.
 *   Outputs: points [P,L,3] fp32 X in the camera-a frame, 0 where a row is not kept (may be NULL); mask
 *   [P,L] uint8 (may be NULL); the kept rows in input order as out_pairs [P,L,2] (-1 padded), out_scores
 *   [P,L] (0 padded), out_counts [P] -- the matcher's list format.
 * Limits: L <= 16384, 0 <= refine_iters <= 100, threshold > 0 and finite, 0 <= max_parallax_cos <= 1,
 * distance_thresh > 0, fx, fy > 0 and finite, cx, cy finite.
 */
int sslam_triangulate(const float* kpts1, int F1, const float* kpts2, int F2, const int32_t* pair_index,
                      int P, int N, int M, const int32_t* pairs, const float* pair_scores,
                      const int32_t* counts, int L, const double* R, const double* t, double fx, double fy,
                      double cx, double cy, double threshold, double max_parallax_cos,
                      double distance_thresh, int refine_iters, float* points, int32_t* out_pairs,
                      float* out_scores, int32_t* out_counts, uint8_t* mask, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Sliding-window bundle adjustment: for each of P windows of W posed frames, the poses of the last
 * W - fixed frames and the points of the window's tracks are refined jointly on the pixel error of every
 * observation, in one launch (one CTA per window), without host synchronisation (capturable in a CUDA
 * graph), without atomics; a window's result does not depend on its position in the batch.
 *   kpts [F,K,2] fp32 pixel bank; frame_index [P,W] int32 slot of each window frame; obs [P,N,W] int32
 *   keypoint of track n in window frame w (-1: none); points [P,N,3] fp32 track points in the world frame;
 *   counts [P] int32 tracks per window; R [P,W,9] row-major, t [P,W,3] double, x_w ~ R_w X + t_w; one
 *   pinhole camera.  The first `fixed` frames of every window are held (2 pins the monocular scale).
 *   Used set, fixed at the start: observation (n, w) is used when its slot and keypoint index are in range,
 *   its keypoint and the point are finite and the depth is > 0; a track is used when n < counts[p] and it
 *   has at least 2 such observations.  Cost: sum of rho(|r|^2) over used observations, r = pi(R_w X + t_w)
 *   - x, rho Huber with threshold `huber` px (inf: least squares), IRLS weight min(1, huber / |r|) at the
 *   linearisation point.  Levenberg-Marquardt (R_w <- Exp(w) R_w, t_w <- t_w + d, X <- X + dX), damping
 *   H_ii (1 + lambda), lambda0 = 1e-3 mean diag(J^T W J) over all free parameters, /10 on an accepted
 *   trial, x10 otherwise; each trial solves the Schur complement on the poses by a dense Cholesky (not
 *   positive definite or a step that is not finite: rejected) and back-substitutes per track; a candidate
 *   with a used observation at depth <= 0 is rejected, a strictly lower cost accepted.  All arithmetic is
 *   double and correctly rounded except Rodrigues' sin / cos; sums run in ascending track, then frame order.
 *   Outputs: R_out, t_out (held frames copied bit for bit); points_out [P,N,3] fp32 (refined for used
 *   tracks, copied otherwise); rms [P,2] double, the RMS pixel error over the used observations before /
 *   after; accepted [P] int32 accepted trials (may be NULL); mask [P,N,W] uint8, used and squared error
 *   < threshold^2 at the end (may be NULL).  A window with a pose that is not finite or an all-zero R, or
 *   without a used track, is returned unchanged with zero rms, accepted and mask.
 *   The workspace (sslam_bundle_adjust_workspace_bytes) holds 49 bytes per track and window.
 * Limits: 2 <= W <= 8 (SSLAM_EUNSUPPORTED above), 1 <= fixed <= W, N <= 65536 (SSLAM_EUNSUPPORTED
 * above), 0 <= refine_iters <= 100, huber > 0, threshold > 0 and finite, fx, fy > 0 and finite, cx, cy
 * finite.
 */
size_t sslam_bundle_adjust_workspace_bytes(int P, int N);
int sslam_bundle_adjust(const float* kpts, int F, int K, const int32_t* frame_index, int P, int W, int N,
                        const int32_t* obs, const float* points, const int32_t* counts, const double* R,
                        const double* t, double fx, double fy, double cx, double cy, int fixed, double huber,
                        double threshold, int refine_iters, double* R_out, double* t_out, float* points_out,
                        double* rms, int32_t* accepted, uint8_t* mask, void* ws, size_t ws_bytes,
                        void* stream);

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
