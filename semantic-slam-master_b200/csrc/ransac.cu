// Geometric verification of padded match lists: batched RANSAC for P pairs at once, against a
// homography (HModel) or a fundamental matrix (FModel).  The three kernels are templates over the model;
// only the minimal solve, the inlier test and the refit's normal rows and post-processing differ.
//
//   ransac_hyp     one thread per (pair, sample): SAMPLE distinct rows drawn by a counter-based
//                  splitmix64 sampler, minimal solve in double -> SLOTS fp32 hypotheses
//   ransac_score   the hot loop (P x SLOTS*iters x n error evaluations): the pair's correspondences are
//                  staged in shared memory tile by tile, warps take hypotheses, lanes stride the points
//   ransac_refit   one CTA per pair: best hypothesis slot (most inliers, lowest slot on ties), least-squares
//                  normalised fit over its inliers (fixed-order double reductions, Jacobi on one
//                  thread), re-score, order-preserving compaction into the matcher's list format
//
// HModel: 4 rows, normalised 4-point DLT, forward transfer error, one slot per sample.
// FModel: 7 rows, normalised 7-point solve — full-pivot elimination of the 7x9 system, real roots of
//   det(F2 + lam (F1 - F2)) by critical-point splitting and 64-step bisection — three slots per sample
//   (3s, 3s+1, 3s+2 in root order, unused slots degenerate), symmetric epipolar error (both squared
//   point-to-line distances < t^2), 8-point refit with rank 2 enforced.
//
// Every result is a function of (inputs, iters, threshold, seed) only: the samples of sample s depend
// on (seed, s, n) and not on the pair's position in the batch, and no reduction uses atomics.
// oracle/geometry.py (H) and oracle/fundamental.py (F) restate the sampler, the minimal solves and the
// scoring operation by operation: the hypothesis path uses only correctly rounded operations
// (__dmul_rn / __dadd_rn / __ddiv_rn / __dsqrt_rn, __fmul_rn / __fadd_rn / __frcp_rn) in fixed orders with
// fixed iteration counts, so CUDA and NumPy agree bit for bit.
#include "common.cuh"

namespace sslam {
namespace {

constexpr int MAX_L = 16384;          // list stride limit (refit flags live in shared memory)
constexpr int MAX_ITERS = 65536;
constexpr int MAX_DRAWS = 32;         // sampler draws per sample (redraws included)
constexpr int HYP_THREADS = 64;
constexpr int SC_THREADS = 256;
constexpr int SC_HYPS = 256;          // hypotheses per scoring CTA (32 per warp)
constexpr int SC_TILE = 4096;         // correspondences staged per tile: 64 KB, three CTAs per SM
constexpr int RF_THREADS = 256;
constexpr double PIVOT_TOL = 1e-8;    // |pivot| of the normalised 8x8 / 7x9 solves, |h33| before scaling
constexpr int BISECT = 64;            // bisection steps per sign-changing bracket of the 7-point cubic
constexpr double SQRT2 = 1.4142135623730951;

// ---------------------------------------------------------------------------- shared pieces
struct RansacParams {
  const float* k1; const float* k2;          // [F1,N,2], [F2,M,2]
  int F1, F2;
  const int32_t* pair_index;                 // [P,2] or null
  int P, N, M;
  const int32_t* pairs; const float* pair_scores; const int32_t* counts;   // [P,L,2], [P,L], [P]
  int L, iters;
  float t2;                                  // threshold^2 rounded to fp32
  u64 seed;
  double* H;                                 // [P,9] or null: the model (H or F)
  int32_t* out_pairs; float* out_scores; int32_t* out_counts; uint8_t* mask;
  // workspace
  int32_t* hyp_count;                        // [P,SLOTS*iters]  inliers per hypothesis slot, -1 degenerate
  int32_t* best;                             // [P]              best slot, -1 none
  uint8_t* hyp_mask;                         // [P,L]            inliers of the best slot
  float* hyp;                                // [P,SLOTS*iters,9]
};

// Rows of pair p, clamped to the list stride; 0 when the pair's frame ids are out of range.
__device__ __forceinline__ int pair_rows(const RansacParams& r, int p, int& a, int& b) {
  a = p; b = p;
  if (r.pair_index) { a = r.pair_index[2 * p]; b = r.pair_index[2 * p + 1]; }
  if (a < 0 || a >= r.F1 || b < 0 || b >= r.F2) return 0;
  return min(max(r.counts[p], 0), r.L);
}

// Correspondence of row k as (x1, y1, x2, y2); NaN (never an inlier, degenerate sample) when the
// row's keypoint indices are out of range.
__device__ __forceinline__ float4 corr(const RansacParams& r, int p, int a, int b, int k) {
  const int2 ij = reinterpret_cast<const int2*>(r.pairs)[(size_t)p * r.L + k];
  if (ij.x < 0 || ij.x >= r.N || ij.y < 0 || ij.y >= r.M) {
    const float nan = __int_as_float(0x7fc00000);
    return make_float4(nan, nan, nan, nan);
  }
  const float2 u = reinterpret_cast<const float2*>(r.k1)[(size_t)a * r.N + ij.x];
  const float2 v = reinterpret_cast<const float2*>(r.k2)[(size_t)b * r.M + ij.y];
  return make_float4(u.x, u.y, v.x, v.y);
}

// Output k (0-based) of the splitmix64 stream seeded with `seed`.
__device__ __forceinline__ u64 splitmix64(u64 seed, u64 k) {
  u64 z = seed + (k + 1) * 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// R distinct rows of [0, n) for sample h: draw c uses output h*MAX_DRAWS + c, a repeat is redrawn.
template <int R>
__device__ __forceinline__ bool sample_rows(u64 seed, int h, int n, int idx[R]) {
  int got = 0;
  for (int c = 0; c < MAX_DRAWS && got < R; ++c) {
    const u64 u = splitmix64(seed, (u64)h * MAX_DRAWS + c);
    const int i = (int)(((u >> 32) * (u64)n) >> 32);
    bool dup = false;
#pragma unroll
    for (int q = 0; q < R; ++q) dup |= (q < got && idx[q] == i);
    if (!dup) {
#pragma unroll
      for (int q = 0; q < R; ++q) if (q == got) idx[q] = i;
      ++got;
    }
  }
  return got == R;
}

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dadd_rn(a, -b); }

// H = T2^-1 . Hn . T1 with T = [[s,0,-s*cx],[0,s,-s*cy],[0,0,1]], then scaled to h33 = 1.
// false when |h33| < PIVOT_TOL or a coefficient is not finite.
__device__ bool denormalise(const double hn[9], double s1, double cx1, double cy1, double s2, double cx2,
                            double cy2, double H[9]) {
  const double tx = dmul(-s1, cx1), ty = dmul(-s1, cy1);
  double m[9];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    m[3 * r + 0] = dmul(hn[3 * r + 0], s1);
    m[3 * r + 1] = dmul(hn[3 * r + 1], s1);
    m[3 * r + 2] = dadd(dadd(dmul(hn[3 * r + 0], tx), dmul(hn[3 * r + 1], ty)), hn[3 * r + 2]);
  }
  const double is2 = __ddiv_rn(1.0, s2);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    H[c] = dadd(dmul(is2, m[c]), dmul(cx2, m[6 + c]));
    H[3 + c] = dadd(dmul(is2, m[3 + c]), dmul(cy2, m[6 + c]));
    H[6 + c] = m[6 + c];
  }
  const double w = H[8];
  if (!(fabs(w) >= PIVOT_TOL)) return false;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 8; ++k) { H[k] = __ddiv_rn(H[k], w); ok &= isfinite(H[k]); }
  H[8] = 1.0;
  return ok;
}

// Centroid and sqrt(2)/mean distance of 4 points; false when they coincide.
__device__ __forceinline__ bool norm4(const double x[4], const double y[4], double& cx, double& cy, double& s) {
  cx = dmul(dadd(dadd(dadd(x[0], x[1]), x[2]), x[3]), 0.25);
  cy = dmul(dadd(dadd(dadd(y[0], y[1]), y[2]), y[3]), 0.25);
  double md = 0.0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const double dx = dsub(x[q], cx), dy = dsub(y[q], cy);
    md = q == 0 ? __dsqrt_rn(dadd(dmul(dx, dx), dmul(dy, dy)))
                : dadd(md, __dsqrt_rn(dadd(dmul(dx, dx), dmul(dy, dy))));
  }
  md = dmul(md, 0.25);
  if (!(md > 0.0)) return false;
  s = __ddiv_rn(SQRT2, md);
  return true;
}

// Normalised 4-point DLT: the 8x8 system with h33 = 1, Gaussian elimination with partial pivoting
// (column c: rows c+1..7 in order, a row whose |entry| is strictly larger than the current pivot's is
// swapped into row c), back substitution, denormalisation.  false marks a degenerate sample.
__device__ bool dlt4(const float4 q[4], double H[9]) {
  double x1[4], y1[4], x2[4], y2[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) { x1[k] = q[k].x; y1[k] = q[k].y; x2[k] = q[k].z; y2[k] = q[k].w; }
  double cx1, cy1, s1, cx2, cy2, s2;
  if (!norm4(x1, y1, cx1, cy1, s1) || !norm4(x2, y2, cx2, cy2, s2)) return false;
  double A[8][9];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double x = dmul(dsub(x1[k], cx1), s1), y = dmul(dsub(y1[k], cy1), s1);
    const double u = dmul(dsub(x2[k], cx2), s2), v = dmul(dsub(y2[k], cy2), s2);
    double* r0 = A[2 * k];
    double* r1 = A[2 * k + 1];
    r0[0] = x; r0[1] = y; r0[2] = 1.0; r0[3] = 0.0; r0[4] = 0.0; r0[5] = 0.0;
    r0[6] = dmul(-u, x); r0[7] = dmul(-u, y); r0[8] = u;
    r1[0] = 0.0; r1[1] = 0.0; r1[2] = 0.0; r1[3] = x; r1[4] = y; r1[5] = 1.0;
    r1[6] = dmul(-v, x); r1[7] = dmul(-v, y); r1[8] = v;
  }
  bool ok = true;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
#pragma unroll
    for (int r = c + 1; r < 8; ++r) {
      const bool sw = fabs(A[r][c]) > fabs(A[c][c]);
#pragma unroll
      for (int k = c; k < 9; ++k) {
        const double t = A[c][k];
        A[c][k] = sw ? A[r][k] : t;
        A[r][k] = sw ? t : A[r][k];
      }
    }
    ok &= fabs(A[c][c]) >= PIVOT_TOL;
#pragma unroll
    for (int r = c + 1; r < 8; ++r) {
      const double f = __ddiv_rn(A[r][c], A[c][c]);
#pragma unroll
      for (int k = c + 1; k < 9; ++k) A[r][k] = dsub(A[r][k], dmul(f, A[c][k]));
    }
  }
  if (!ok) return false;
  double hn[9];
  hn[8] = 1.0;
#pragma unroll
  for (int c = 7; c >= 0; --c) {
    double acc = A[c][8];
#pragma unroll
    for (int k = c + 1; k < 8; ++k) acc = dsub(acc, dmul(A[c][k], hn[k]));
    hn[c] = __ddiv_rn(acc, A[c][c]);
  }
  return denormalise(hn, s1, cx1, cy1, s2, cx2, cy2, H);
}

// Forward transfer error test in fp32: u, v, w = H.(x1, y1, 1); (u/w, v/w) as u*(1/w), v*(1/w).
__device__ __forceinline__ bool is_inlier(const float h[9], float4 q, float t2) {
  const float u = __fadd_rn(__fadd_rn(__fmul_rn(h[0], q.x), __fmul_rn(h[1], q.y)), h[2]);
  const float v = __fadd_rn(__fadd_rn(__fmul_rn(h[3], q.x), __fmul_rn(h[4], q.y)), h[5]);
  const float w = __fadd_rn(__fadd_rn(__fmul_rn(h[6], q.x), __fmul_rn(h[7], q.y)), h[8]);
  const float iw = __frcp_rn(w);
  const float dx = __fsub_rn(__fmul_rn(u, iw), q.z);
  const float dy = __fsub_rn(__fmul_rn(v, iw), q.w);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) < t2;
}

// Cyclic Jacobi on a symmetric NxN (one thread, shared memory); returns the eigenvector of the
// smallest eigenvalue in v_out.
template <int N>
__device__ void jacobi_smallest(double* A, double* V, double* v_out) {
  for (int i = 0; i < N * N; ++i) V[i] = (i % (N + 1) == 0) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 50; ++sweep) {
    double off = 0.0, tot = 0.0;
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) {
        const double e = A[N * i + j] * A[N * i + j];
        tot += e;
        if (i != j) off += e;
      }
    if (!(off > 1e-30 * tot)) break;
    for (int p = 0; p < N - 1; ++p)
      for (int q = p + 1; q < N; ++q) {
        const double apq = A[N * p + q];
        if (apq == 0.0) continue;
        const double theta = (A[N * q + q] - A[N * p + p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < N; ++k) {                    // A <- A J (columns p, q)
          const double akp = A[N * k + p], akq = A[N * k + q];
          A[N * k + p] = c * akp - s * akq;
          A[N * k + q] = s * akp + c * akq;
        }
        for (int k = 0; k < N; ++k) {                    // A <- J^T A (rows p, q)
          const double apk = A[N * p + k], aqk = A[N * q + k];
          A[N * p + k] = c * apk - s * aqk;
          A[N * q + k] = s * apk + c * aqk;
        }
        for (int k = 0; k < N; ++k) {                    // V <- V J
          const double vkp = V[N * k + p], vkq = V[N * k + q];
          V[N * k + p] = c * vkp - s * vkq;
          V[N * k + q] = s * vkp + c * vkq;
        }
      }
  }
  int m = 0;
  for (int i = 1; i < N; ++i) if (A[(N + 1) * i] < A[(N + 1) * m]) m = i;
  for (int k = 0; k < N; ++k) v_out[k] = V[N * k + m];
}

// ---------------------------------------------------------------------------- homography model
// Slots of sample s: bit k of solve()'s result marks slot k valid.  accumulate() adds one inlier's
// normal-matrix terms (upper triangle, 45 sums); finish() turns the smallest eigenvector of the normal
// matrix into the model (thread 0; A, V: 81-double shared scratch).
struct HModel {
  static constexpr int SAMPLE = 4, SLOTS = 1, MIN_FIT = 4;
  __device__ static int solve(const float4 q[SAMPLE], double H[SLOTS][9]) { return dlt4(q, H[0]) ? 1 : 0; }
  __device__ static bool inlier(const float h[9], float4 q, float t2) { return is_inlier(h, q, t2); }
  __device__ static void accumulate(double x, double y, double u, double v, double (&nm)[45]) {
    const double r0[9] = {x, y, 1.0, 0.0, 0.0, 0.0, -u * x, -u * y, -u};
    const double r1[9] = {0.0, 0.0, 0.0, x, y, 1.0, -v * x, -v * y, -v};
    int t = 0;
#pragma unroll
    for (int i = 0; i < 9; ++i)
#pragma unroll
      for (int j = i; j < 9; ++j, ++t) nm[t] = dadd(nm[t], dadd(dmul(r0[i], r0[j]), dmul(r1[i], r1[j])));
  }
  __device__ static bool finish(const double hn[9], double s1, double cx1, double cy1, double s2, double cx2,
                                double cy2, double H[9], double*, double*) {
    return denormalise(hn, s1, cx1, cy1, s2, cx2, cy2, H);
  }
};

// ---------------------------------------------------------------------------- fundamental model
// Centroid and sqrt(2)/mean distance of 7 points; false when they coincide.
__device__ __forceinline__ bool norm7(const double x[7], const double y[7], double& cx, double& cy, double& s) {
  double sx = x[0], sy = y[0];
#pragma unroll
  for (int q = 1; q < 7; ++q) { sx = dadd(sx, x[q]); sy = dadd(sy, y[q]); }
  cx = __ddiv_rn(sx, 7.0);
  cy = __ddiv_rn(sy, 7.0);
  double md = 0.0;
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    const double dx = dsub(x[q], cx), dy = dsub(y[q], cy);
    md = q == 0 ? __dsqrt_rn(dadd(dmul(dx, dx), dmul(dy, dy)))
                : dadd(md, __dsqrt_rn(dadd(dmul(dx, dx), dmul(dy, dy))));
  }
  md = __ddiv_rn(md, 7.0);
  if (!(md > 0.0)) return false;
  s = __ddiv_rn(SQRT2, md);
  return true;
}

// Unit Frobenius norm, then the largest-|entry| element (lowest index on ties) made positive.
// false when the norm is zero or a coefficient is not finite.
__device__ bool unit_sign(double F[9]) {
  double n2 = dmul(F[0], F[0]);
#pragma unroll
  for (int k = 1; k < 9; ++k) n2 = dadd(n2, dmul(F[k], F[k]));
  const double nrm = __dsqrt_rn(n2);
  if (!(nrm > 0.0) || !isfinite(nrm)) return false;
#pragma unroll
  for (int k = 0; k < 9; ++k) F[k] = __ddiv_rn(F[k], nrm);
  int big = 0;
#pragma unroll
  for (int k = 1; k < 9; ++k) big = fabs(F[k]) > fabs(F[big]) ? k : big;
  const bool neg = F[big] < 0.0;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 9; ++k) { F[k] = neg ? -F[k] : F[k]; ok &= isfinite(F[k]); }
  return ok;
}

// F = T2^T . Fn . T1 with T = [[s,0,-s*cx],[0,s,-s*cy],[0,0,1]], then unit_sign.
__device__ bool denormalise_f(const double fn[9], double s1, double cx1, double cy1, double s2, double cx2,
                              double cy2, double F[9]) {
  const double tx = dmul(-s1, cx1), ty = dmul(-s1, cy1);
  double m[9];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    m[3 * r + 0] = dmul(fn[3 * r + 0], s1);
    m[3 * r + 1] = dmul(fn[3 * r + 1], s1);
    m[3 * r + 2] = dadd(dadd(dmul(fn[3 * r + 0], tx), dmul(fn[3 * r + 1], ty)), fn[3 * r + 2]);
  }
  const double ux = dmul(-s2, cx2), uy = dmul(-s2, cy2);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    F[c] = dmul(s2, m[c]);
    F[3 + c] = dmul(s2, m[3 + c]);
    F[6 + c] = dadd(dadd(dmul(ux, m[c]), dmul(uy, m[3 + c])), m[6 + c]);
  }
  return unit_sign(F);
}

// r0 . (r1 x r2) in fixed order.
__device__ __forceinline__ double det3(const double* r0, const double* r1, const double* r2) {
  const double k0 = dsub(dmul(r1[1], r2[2]), dmul(r1[2], r2[1]));
  const double k1 = dsub(dmul(r1[2], r2[0]), dmul(r1[0], r2[2]));
  const double k2 = dsub(dmul(r1[0], r2[1]), dmul(r1[1], r2[0]));
  return dadd(dadd(dmul(r0[0], k0), dmul(r0[1], k1)), dmul(r0[2], k2));
}

__device__ __forceinline__ double poly3(double a3, double a2, double a1, double a0, double x) {
  return dadd(dmul(dadd(dmul(dadd(dmul(a3, x), a2), x), a1), x), a0);
}

// Real roots of a3 x^3 + a2 x^2 + a1 x + a0 on [-1, 1] (closed) or (-1, 1), ascending, into out[7].
// The interval is split at the real critical points (quadratic formula, correctly rounded sqrt; a
// critical point outside the open interval is dropped); a breakpoint where the polynomial is exactly 0
// is a root, and a bracket with a strict sign change is bisected BISECT times.  Not inlined, like
// seven_point: inlined, it makes seven_point spill.
__device__ __noinline__ int cubic_roots(double a3, double a2, double a1, double a0, bool closed, double out[7]) {
  const double lo = -1.0, hi = 1.0;
  const double t3 = dmul(3.0, a3);
  const double disc = dsub(dmul(a2, a2), dmul(t3, a1));
  const bool quad = a3 != 0.0 && disc >= 0.0;
  const bool lin = a3 == 0.0 && a2 != 0.0;
  double cA = 0.0, cB = 0.0;
  if (quad) {
    const double sq = __dsqrt_rn(disc);
    const double r1 = __ddiv_rn(dsub(-a2, sq), t3), r2 = __ddiv_rn(dadd(-a2, sq), t3);
    cA = r1 < r2 ? r1 : r2;
    cB = r1 < r2 ? r2 : r1;
  } else if (lin) {
    cA = __ddiv_rn(-a1, dmul(2.0, a2));
  }
  const bool vA = (quad || lin) && cA > lo && cA < hi;
  const bool vB = quad && disc > 0.0 && cB > lo && cB < hi;
  double pt[4];
  pt[0] = lo;
  pt[1] = vA ? cA : lo;
  pt[2] = vB ? cB : pt[1];
  pt[3] = hi;
  const bool pv[4] = {true, vA, vB, true};
  double g[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) g[i] = poly3(a3, a2, a1, a0, pt[i]);
  int cnt = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (pv[i] && g[i] == 0.0 && (closed || (i > 0 && i < 3))) out[cnt++] = pt[i];
    if (i < 3 && ((g[i] < 0.0 && g[i + 1] > 0.0) || (g[i] > 0.0 && g[i + 1] < 0.0))) {
      double a = pt[i], b = pt[i + 1];
      const bool neg = g[i] < 0.0;
      for (int it = 0; it < BISECT; ++it) {
        const double m = dmul(dadd(a, b), 0.5);
        if ((poly3(a3, a2, a1, a0, m) < 0.0) == neg) a = m; else b = m;
      }
      out[cnt++] = dmul(dadd(a, b), 0.5);
    }
  }
  return cnt;
}

// Null vector of the reduced 7x9 system with free column j set to 1 (the other free column 0), by
// back substitution in fixed order.
__device__ __forceinline__ void back_substitute(const double (&A)[7][9], const int (&piv)[7], int j, double f[9]) {
#pragma unroll
  for (int k = 0; k < 9; ++k) f[k] = 0.0;
  f[j] = 1.0;
  for (int r = 6; r >= 0; --r) {
    double acc = A[r][j];
    for (int r2 = r + 1; r2 < 7; ++r2) acc = dadd(acc, dmul(A[r][piv[r2]], f[piv[r2]]));
    f[piv[r]] = __ddiv_rn(-acc, A[r][piv[r]]);
  }
}

// Normalised 7-point solve.  Rows [u x, u y, u, v x, v y, v, x, y, 1] (x1 = (x, y), x2 = (u, v)),
// Gaussian elimination with full pivoting (largest |entry| of the remaining submatrix, lowest (row,
// column) on ties; rows below the pivot reduced in the columns that have not pivoted); a pivot below
// 1e-8 marks the sample degenerate (with full pivoting the 7th is the first to fall: 7 correspondences
// related by one homography give a rank-6 system).  The two free columns j1 < j2 give f1, f2; the real
// roots of det(F2 + lam D), D = F1 - F2, fill the slots in order: lam in [-1, 1] from p(lam), then
// mu = 1/lam in (-1, 1) from q(mu) = mu^3 p(1/mu) as mu F2 + D (mu = 0 is D).  A root whose F is not
// finite or has zero norm leaves its slot degenerate.
// Not inlined: inlined into ransac_refit_kernel it makes ptxas cap that kernel at 128 registers and spill.
__device__ __noinline__ int seven_point(const float4 q[7], double F[3][9]) {
  double x1[7], y1[7], x2[7], y2[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) { x1[k] = q[k].x; y1[k] = q[k].y; x2[k] = q[k].z; y2[k] = q[k].w; }
  double cx1, cy1, s1, cx2, cy2, s2;
  if (!norm7(x1, y1, cx1, cy1, s1) || !norm7(x2, y2, cx2, cy2, s2)) return 0;
  double A[7][9];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const double x = dmul(dsub(x1[k], cx1), s1), y = dmul(dsub(y1[k], cy1), s1);
    const double u = dmul(dsub(x2[k], cx2), s2), v = dmul(dsub(y2[k], cy2), s2);
    A[k][0] = dmul(u, x); A[k][1] = dmul(u, y); A[k][2] = u;
    A[k][3] = dmul(v, x); A[k][4] = dmul(v, y); A[k][5] = v;
    A[k][6] = x; A[k][7] = y; A[k][8] = 1.0;
  }
  bool used[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) used[c] = false;
  int piv[7];
  for (int r = 0; r < 7; ++r) {
    double bv = -1.0;
    int bi = r, bc = 0;
    for (int i = r; i < 7; ++i)
      for (int c = 0; c < 9; ++c) {
        const double v = used[c] ? -1.0 : fabs(A[i][c]);
        if (v > bv) { bv = v; bi = i; bc = c; }
      }
    for (int k = 0; k < 9; ++k) {
      const double t = A[r][k];
      A[r][k] = A[bi][k];
      A[bi][k] = t;
    }
    used[bc] = true;
    piv[r] = bc;
    const double pv = A[r][bc];
    if (!(fabs(pv) >= PIVOT_TOL)) return 0;
    for (int i = r + 1; i < 7; ++i) {
      const double f = __ddiv_rn(A[i][bc], pv);
      for (int k = 0; k < 9; ++k)
        if (!used[k]) A[i][k] = dsub(A[i][k], dmul(f, A[r][k]));
    }
  }
  int j1 = -1, j2 = -1;
  for (int c = 0; c < 9; ++c)
    if (!used[c]) { if (j1 < 0) j1 = c; else j2 = c; }
  double f1[9], f2[9], d[9];
  back_substitute(A, piv, j1, f1);
  back_substitute(A, piv, j2, f2);
#pragma unroll
  for (int k = 0; k < 9; ++k) d[k] = dsub(f1[k], f2[k]);
  const double c0 = det3(f2, f2 + 3, f2 + 6);
  const double c1 = dadd(dadd(det3(d, f2 + 3, f2 + 6), det3(f2, d + 3, f2 + 6)), det3(f2, f2 + 3, d + 6));
  const double c2 = dadd(dadd(det3(f2, d + 3, d + 6), det3(d, f2 + 3, d + 6)), det3(d, d + 3, f2 + 6));
  const double c3 = det3(d, d + 3, d + 6);
  double root[7];
  int slots = 0, valid = 0;
  for (int pass = 0; pass < 2; ++pass) {
    const int nr = pass == 0 ? cubic_roots(c3, c2, c1, c0, true, root) : cubic_roots(c0, c1, c2, c3, false, root);
    for (int i = 0; i < nr && slots < 3; ++i, ++slots) {
      double fn[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) fn[k] = pass == 0 ? dadd(f2[k], dmul(root[i], d[k])) : dadd(dmul(root[i], f2[k]), d[k]);
      if (denormalise_f(fn, s1, cx1, cy1, s2, cx2, cy2, F[slots])) valid |= 1 << slots;
    }
  }
  return valid;
}

// Symmetric epipolar test in fp32 (cv2's FM_RANSAC error): the squared distance of x2 to the line
// F.x1 and of x1 to the line F^T.x2, each as d*d * rcp(a*a + b*b); both must be < t2, so a NaN (an
// undefined line) is an outlier.
__device__ __forceinline__ bool epi_inlier(const float f[9], float4 q, float t2) {
  const float a2 = __fadd_rn(__fadd_rn(__fmul_rn(f[0], q.x), __fmul_rn(f[1], q.y)), f[2]);
  const float b2 = __fadd_rn(__fadd_rn(__fmul_rn(f[3], q.x), __fmul_rn(f[4], q.y)), f[5]);
  const float c2 = __fadd_rn(__fadd_rn(__fmul_rn(f[6], q.x), __fmul_rn(f[7], q.y)), f[8]);
  const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(q.z, a2), __fmul_rn(q.w, b2)), c2);
  const float e2 = __fmul_rn(__fmul_rn(d2, d2), __frcp_rn(__fadd_rn(__fmul_rn(a2, a2), __fmul_rn(b2, b2))));
  const float a1 = __fadd_rn(__fadd_rn(__fmul_rn(f[0], q.z), __fmul_rn(f[3], q.w)), f[6]);
  const float b1 = __fadd_rn(__fadd_rn(__fmul_rn(f[1], q.z), __fmul_rn(f[4], q.w)), f[7]);
  const float c1 = __fadd_rn(__fadd_rn(__fmul_rn(f[2], q.z), __fmul_rn(f[5], q.w)), f[8]);
  const float d1 = __fadd_rn(__fadd_rn(__fmul_rn(q.x, a1), __fmul_rn(q.y, b1)), c1);
  const float e1 = __fmul_rn(__fmul_rn(d1, d1), __frcp_rn(__fadd_rn(__fmul_rn(a1, a1), __fmul_rn(b1, b1))));
  return e1 < t2 && e2 < t2;
}

struct FModel {
  static constexpr int SAMPLE = 7, SLOTS = 3, MIN_FIT = 8;
  __device__ static int solve(const float4 q[SAMPLE], double F[SLOTS][9]) { return seven_point(q, F); }
  __device__ static bool inlier(const float f[9], float4 q, float t2) { return epi_inlier(f, q, t2); }
  __device__ static void accumulate(double x, double y, double u, double v, double (&nm)[45]) {
    const double r0[9] = {u * x, u * y, u, v * x, v * y, v, x, y, 1.0};
    int t = 0;
#pragma unroll
    for (int i = 0; i < 9; ++i)
#pragma unroll
      for (int j = i; j < 9; ++j, ++t) nm[t] = dadd(nm[t], dmul(r0[i], r0[j]));
  }
  // Rank 2 as Fn - (Fn.v3).v3^T, v3 the smallest eigenvector of Fn^T.Fn (3x3 Jacobi), then denormalise.
  __device__ static bool finish(const double fn[9], double s1, double cx1, double cy1, double s2, double cx2,
                                double cy2, double F[9], double* A, double* V) {
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) A[3 * i + j] = fn[i] * fn[j] + fn[3 + i] * fn[3 + j] + fn[6 + i] * fn[6 + j];
    double v3[3], fr[9];
    jacobi_smallest<3>(A, V, v3);
    for (int i = 0; i < 3; ++i) {
      const double w = fn[3 * i] * v3[0] + fn[3 * i + 1] * v3[1] + fn[3 * i + 2] * v3[2];
      for (int j = 0; j < 3; ++j) fr[3 * i + j] = fn[3 * i + j] - w * v3[j];
    }
    return denormalise_f(fr, s1, cx1, cy1, s2, cx2, cy2, F);
  }
};

// ---------------------------------------------------------------------------- shared by both models
// Slots of sample s of pair p as doubles: bit k set when slot k holds a model.
template <class M>
__device__ __forceinline__ int sample_hyps(const RansacParams& r, int p, int a, int b, int n, int s,
                                           double Hs[M::SLOTS][9]) {
  int idx[M::SAMPLE];
#pragma unroll
  for (int k = 0; k < M::SAMPLE; ++k) idx[k] = -1;
  if (n < M::SAMPLE || !sample_rows<M::SAMPLE>(r.seed, s, n, idx)) return 0;
  float4 q[M::SAMPLE];
#pragma unroll
  for (int k = 0; k < M::SAMPLE; ++k) q[k] = corr(r, p, a, b, idx[k]);
  return M::solve(q, Hs);
}

// Hypothesis slot h of pair p as doubles (false: degenerate).
template <class M>
__device__ bool slot_hypothesis(const RansacParams& r, int p, int a, int b, int n, int h, double H[9]) {
  double Hs[M::SLOTS][9];
  const int k = h % M::SLOTS;
  if (!((sample_hyps<M>(r, p, a, b, n, h / M::SLOTS, Hs) >> k) & 1)) return false;
  for (int j = 0; j < 9; ++j) H[j] = Hs[k][j];
  return true;
}

// ---------------------------------------------------------------------------- kernels
template <class M>
__global__ void __launch_bounds__(HYP_THREADS) ransac_hyp_kernel(RansacParams r) {
  const int p = blockIdx.x;
  const int s = blockIdx.y * HYP_THREADS + threadIdx.x;
  if (s >= r.iters) return;
  int a, b;
  const int n = pair_rows(r, p, a, b);
  double H[M::SLOTS][9];
  const int ok = sample_hyps<M>(r, p, a, b, n, s, H);
#pragma unroll
  for (int j = 0; j < M::SLOTS; ++j) {
    const size_t h = ((size_t)p * r.iters + s) * M::SLOTS + j;
    const bool v = (ok >> j) & 1;
    float* o = r.hyp + h * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) o[k] = v ? __double2float_rn(H[j][k]) : 0.f;
    r.hyp_count[h] = v ? 0 : -1;
  }
}

template <class M>
__global__ void __launch_bounds__(SC_THREADS) ransac_score_kernel(RansacParams r, int tile) {
  extern __shared__ float4 pts[];
  __shared__ float hs[SC_HYPS][9];
  __shared__ int cnt[SC_HYPS];
  const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slots = M::SLOTS * r.iters;
  const int h0 = blockIdx.y * SC_HYPS;
  const int nh = min(SC_HYPS, slots - h0);
  int a, b;
  const int n = pair_rows(r, p, a, b);
  if (n < M::SAMPLE) return;                           // every hypothesis of the pair is degenerate
  const size_t base = (size_t)p * slots + h0;
  for (int t = tid; t < nh * 9; t += SC_THREADS) hs[t / 9][t % 9] = r.hyp[base * 9 + t];
  for (int t = tid; t < nh; t += SC_THREADS) cnt[t] = r.hyp_count[base + t];
  for (int k0 = 0; k0 < n; k0 += tile) {
    const int nt = min(tile, n - k0);
    __syncthreads();
    for (int k = tid; k < nt; k += SC_THREADS) pts[k] = corr(r, p, a, b, k0 + k);
    __syncthreads();
    for (int hl = warp; hl < nh; hl += SC_THREADS / 32) {
      if (cnt[hl] < 0) continue;
      float h[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) h[k] = hs[hl][k];
      int c = 0;
      for (int k0 = 0; k0 < nt; k0 += 32) {              // warp-uniform bound: every lane votes
        const int k = k0 + lane;
        c += __popc(__ballot_sync(0xffffffffu, k < nt && M::inlier(h, pts[k], r.t2)));
      }
      if (lane == 0) cnt[hl] += c;
    }
  }
  __syncthreads();
  for (int t = tid; t < nh; t += SC_THREADS) r.hyp_count[base + t] = cnt[t];
}

// Fixed-order block sum of R doubles per thread: warp butterflies, then warps in order.
template <int R>
__device__ __forceinline__ void block_sum(double (&v)[R], double* red /* [RF_THREADS/32][R] */,
                                          double* out /* [R] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < R; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = dadd(x, __shfl_xor_sync(0xffffffffu, x, o));
    if (lane == 0) red[warp * R + i] = x;
  }
  __syncthreads();
  if (threadIdx.x < R) {
    double s = red[threadIdx.x];
    for (int w = 1; w < RF_THREADS / 32; ++w) s = dadd(s, red[w * R + threadIdx.x]);
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

template <class M>
__global__ void __launch_bounds__(RF_THREADS) ransac_refit_kernel(RansacParams r) {
  __shared__ uint8_t flag[MAX_L];
  __shared__ double red[(RF_THREADS / 32) * 45];
  __shared__ double sum[45];
  __shared__ double Aj[81], Vj[81];
  __shared__ double Hs[2][9];                       // [0] best hypothesis, [1] refit
  __shared__ float hf[9];
  __shared__ int scan[RF_THREADS];
  __shared__ unsigned long long bkey[RF_THREADS / 32];
  __shared__ int s_best, s_ok, s_total;
  const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int a, b;
  const int n = pair_rows(r, p, a, b);
  const int slots = M::SLOTS * r.iters;

  // ---- best hypothesis: most inliers, lowest slot on ties
  unsigned long long key = 0;
  if (n >= M::SAMPLE)
    for (int h = tid; h < slots; h += RF_THREADS) {
      const int c = r.hyp_count[(size_t)p * slots + h];
      const unsigned long long k = ((unsigned long long)(unsigned)(c + 1) << 32) | (0xffffffffu - (unsigned)h);
      key = k > key ? k : key;
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long k = __shfl_xor_sync(0xffffffffu, key, o);
    key = k > key ? k : key;
  }
  if (lane == 0) bkey[warp] = key;
  __syncthreads();
  if (tid == 0) {
    unsigned long long k = 0;
    for (int w = 0; w < RF_THREADS / 32; ++w) k = bkey[w] > k ? bkey[w] : k;
    const int best = (k >> 32) == 0 ? -1 : (int)(0xffffffffu - (unsigned)(k & 0xffffffffu));
    s_ok = best >= 0 && slot_hypothesis<M>(r, p, a, b, n, best, Hs[0]);
    s_best = s_ok ? best : -1;
    if (s_ok)
      for (int k2 = 0; k2 < 9; ++k2) hf[k2] = __double2float_rn(Hs[0][k2]);
  }
  __syncthreads();
  const bool have = s_ok;
  uint8_t* hm = r.hyp_mask + (size_t)p * r.L;
  int m = 0;                                        // inliers of the best hypothesis (this thread's rows)
  for (int k = tid; k < r.L; k += RF_THREADS) {
    const bool in = have && k < n && M::inlier(hf, corr(r, p, a, b, k), r.t2);
    flag[k] = in;
    hm[k] = in;
    m += in;
  }
  m = block_reduce_sum(m, scan);                    // scan[] doubles as the reduction scratch (>= 33)

  // ---- refit over the best hypothesis's inliers (normalised least squares)
  bool use_refit = false;
  if (have && m >= M::MIN_FIT) {
    double c4[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k = tid; k < n; k += RF_THREADS)
      if (flag[k]) {
        const float4 q = corr(r, p, a, b, k);
        c4[0] = dadd(c4[0], q.x); c4[1] = dadd(c4[1], q.y); c4[2] = dadd(c4[2], q.z); c4[3] = dadd(c4[3], q.w);
      }
    block_sum<4>(c4, red, sum);
    const double cx1 = sum[0] / m, cy1 = sum[1] / m, cx2 = sum[2] / m, cy2 = sum[3] / m;
    double d2[2] = {0.0, 0.0};
    for (int k = tid; k < n; k += RF_THREADS)
      if (flag[k]) {
        const float4 q = corr(r, p, a, b, k);
        d2[0] = dadd(d2[0], sqrt((q.x - cx1) * (q.x - cx1) + (q.y - cy1) * (q.y - cy1)));
        d2[1] = dadd(d2[1], sqrt((q.z - cx2) * (q.z - cx2) + (q.w - cy2) * (q.w - cy2)));
      }
    block_sum<2>(d2, red, sum);
    const double md1 = sum[0] / m, md2 = sum[1] / m;
    if (md1 > 0.0 && md2 > 0.0) {
      const double s1 = SQRT2 / md1, s2 = SQRT2 / md2;
      double nm[45];
#pragma unroll
      for (int i = 0; i < 45; ++i) nm[i] = 0.0;
      for (int k = tid; k < n; k += RF_THREADS)
        if (flag[k]) {
          const float4 q = corr(r, p, a, b, k);
          const double x = (q.x - cx1) * s1, y = (q.y - cy1) * s1;
          const double u = (q.z - cx2) * s2, v = (q.w - cy2) * s2;
          M::accumulate(x, y, u, v, nm);
        }
      block_sum<45>(nm, red, sum);
      if (tid == 0) {
        int t = 0;
        for (int i = 0; i < 9; ++i)
          for (int j = i; j < 9; ++j, ++t) Aj[9 * i + j] = Aj[9 * j + i] = sum[t];
        double hn[9];
        jacobi_smallest<9>(Aj, Vj, hn);
        s_ok = M::finish(hn, s1, cx1, cy1, s2, cx2, cy2, Hs[1], Aj, Vj);
        if (s_ok)
          for (int k2 = 0; k2 < 9; ++k2) hf[k2] = __double2float_rn(Hs[1][k2]);
      }
      __syncthreads();
      if (s_ok) {
        int c = 0;
        for (int k = tid; k < n; k += RF_THREADS) c += M::inlier(hf, corr(r, p, a, b, k), r.t2);
        c = block_reduce_sum(c, scan);
        use_refit = c >= m;
      }
    }
  }
  __syncthreads();
  if (use_refit)
    for (int k = tid; k < n; k += RF_THREADS) flag[k] = M::inlier(hf, corr(r, p, a, b, k), r.t2);
  if (tid == 0) r.best[p] = s_best;
  if (r.H && tid < 9) r.H[9 * (size_t)p + tid] = have ? Hs[use_refit ? 1 : 0][tid] : 0.0;

  // ---- order-preserving compaction of the kept rows (matcher list format)
  __syncthreads();
  const int seg = (n + RF_THREADS - 1) / RF_THREADS;
  const int beg = min(n, tid * seg), end = min(n, beg + seg);
  int cnt = 0;
  for (int k = beg; k < end; ++k) cnt += flag[k];
  scan[tid] = cnt;
  __syncthreads();
  for (int o = 1; o < RF_THREADS; o <<= 1) {
    const int v = (tid >= o) ? scan[tid - o] : 0;
    __syncthreads();
    scan[tid] += v;
    __syncthreads();
  }
  int pos = scan[tid] - cnt;
  if (tid == RF_THREADS - 1) s_total = scan[RF_THREADS - 1];
  __syncthreads();
  const int total = s_total;
  const int2* in_pr = reinterpret_cast<const int2*>(r.pairs) + (size_t)p * r.L;
  const float* in_sc = r.pair_scores + (size_t)p * r.L;
  int2* pr = reinterpret_cast<int2*>(r.out_pairs) + (size_t)p * r.L;
  float* ps = r.out_scores + (size_t)p * r.L;
  for (int k = beg; k < end; ++k)
    if (flag[k]) { pr[pos] = in_pr[k]; ps[pos] = in_sc[k]; ++pos; }
  for (int k = total + tid; k < r.L; k += RF_THREADS) { pr[k] = make_int2(-1, -1); ps[k] = 0.f; }
  if (r.mask)
    for (int k = tid; k < r.L; k += RF_THREADS) r.mask[(size_t)p * r.L + k] = k < n ? flag[k] : 0;
  if (tid == 0) r.out_counts[p] = total;
}

struct WsLayout { size_t count, best, mask, hyp, total; };

WsLayout ws_layout(int P, int L, int iters, int slots_per_sample) {
  const size_t slots = (size_t)iters * slots_per_sample;
  WsLayout w;
  w.count = 0;
  w.best = align_up((size_t)P * slots * 4, 256);
  w.mask = w.best + align_up((size_t)P * 4, 256);
  w.hyp = w.mask + align_up((size_t)P * L, 256);
  w.total = w.hyp + align_up((size_t)P * slots * 9 * 4, 256);
  return w;
}

template <class M>
size_t workspace_bytes(int P, int L, int iters) {
  if (P <= 0 || L < 0 || iters <= 0) return 0;
  return ws_layout(P, L, iters, M::SLOTS).total;
}

template <class Model>
int ransac(const float* kpts1, int F1, const float* kpts2, int F2, const int32_t* pair_index, int P, int N, int M,
           const int32_t* pairs, const float* pair_scores, const int32_t* counts, int L, int iters, double threshold,
           uint64_t seed, double* H, int32_t* out_pairs, float* out_scores, int32_t* out_counts,
           uint8_t* inlier_mask, void* ws, size_t ws_bytes, void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  SSLAM_REQUIRE(P >= 0 && N >= 0 && M >= 0 && L >= 0, SSLAM_EINVAL, "ransac: bad size");
  SSLAM_REQUIRE(L <= MAX_L, SSLAM_EINVAL, "ransac: list stride %d > %d", L, MAX_L);
  SSLAM_REQUIRE(iters >= 1 && iters <= MAX_ITERS, SSLAM_EINVAL, "ransac: iters=%d (need 1..%d)", iters, MAX_ITERS);
  SSLAM_REQUIRE(threshold > 0.0 && isfinite(threshold), SSLAM_EINVAL, "ransac: threshold must be > 0");
  if (P == 0) return SSLAM_OK;
  SSLAM_REQUIRE(kpts1 && kpts2 && pairs && pair_scores && counts && out_pairs && out_scores && out_counts && ws,
                SSLAM_EINVAL, "ransac: null pointer");
  SSLAM_REQUIRE(F1 > 0 && F2 > 0 && (pair_index || (F1 >= P && F2 >= P)), SSLAM_EINVAL,
                "ransac: banks hold %d / %d sets but %d implicit pairs were requested", F1, F2, P);
  const WsLayout w = ws_layout(P, L, iters, Model::SLOTS);
  SSLAM_REQUIRE(ws_bytes >= w.total, SSLAM_EWORKSPACE, "ransac: workspace %zu < %zu", ws_bytes, w.total);
  char* base = static_cast<char*>(ws);
  RansacParams r{kpts1, kpts2, F1, F2, pair_index, P, N, M, pairs, pair_scores, counts, L, iters,
                 (float)(threshold * threshold), (u64)seed, H, out_pairs, out_scores, out_counts, inlier_mask,
                 reinterpret_cast<int32_t*>(base + w.count), reinterpret_cast<int32_t*>(base + w.best),
                 reinterpret_cast<uint8_t*>(base + w.mask), reinterpret_cast<float*>(base + w.hyp)};
  const int tile = L < 1 ? 1 : (L < SC_TILE ? L : SC_TILE);
  const size_t smem = (size_t)tile * sizeof(float4);
  const int score_ctas = (Model::SLOTS * iters + SC_HYPS - 1) / SC_HYPS;
  static DeviceOnce once;
  if (once.first_use())
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(ransac_score_kernel<Model>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(SC_TILE * sizeof(float4))));
  SSLAM_LAUNCH(KK_RANSAC_HYP, stream,
               ransac_hyp_kernel<Model><<<dim3(P, (iters + HYP_THREADS - 1) / HYP_THREADS), HYP_THREADS, 0,
                                          stream>>>(r));
  SSLAM_LAUNCH(KK_RANSAC_SCORE, stream,
               ransac_score_kernel<Model><<<dim3(P, score_ctas), SC_THREADS, smem, stream>>>(r, tile));
  SSLAM_LAUNCH(KK_RANSAC_REFIT, stream, ransac_refit_kernel<Model><<<P, RF_THREADS, 0, stream>>>(r));
  return SSLAM_OK;
}

}  // namespace
}  // namespace sslam

using namespace sslam;

extern "C" size_t sslam_ransac_workspace_bytes(int P, int L, int iters) {
  return workspace_bytes<HModel>(P, L, iters);
}

extern "C" size_t sslam_ransac_fundamental_workspace_bytes(int P, int L, int iters) {
  return workspace_bytes<FModel>(P, L, iters);
}

extern "C" int sslam_ransac_homography(const float* kpts1, int F1, const float* kpts2, int F2,
                                       const int32_t* pair_index, int P, int N, int M, const int32_t* pairs,
                                       const float* pair_scores, const int32_t* counts, int L, int iters,
                                       double threshold, uint64_t seed, double* H, int32_t* out_pairs,
                                       float* out_scores, int32_t* out_counts, uint8_t* inlier_mask, void* ws,
                                       size_t ws_bytes, void* stream) {
  return ransac<HModel>(kpts1, F1, kpts2, F2, pair_index, P, N, M, pairs, pair_scores, counts, L, iters, threshold,
                        seed, H, out_pairs, out_scores, out_counts, inlier_mask, ws, ws_bytes, stream);
}

extern "C" int sslam_ransac_fundamental(const float* kpts1, int F1, const float* kpts2, int F2,
                                        const int32_t* pair_index, int P, int N, int M, const int32_t* pairs,
                                        const float* pair_scores, const int32_t* counts, int L, int iters,
                                        double threshold, uint64_t seed, double* F, int32_t* out_pairs,
                                        float* out_scores, int32_t* out_counts, uint8_t* inlier_mask, void* ws,
                                        size_t ws_bytes, void* stream) {
  return ransac<FModel>(kpts1, F1, kpts2, F2, pair_index, P, N, M, pairs, pair_scores, counts, L, iters, threshold,
                        seed, F, out_pairs, out_scores, out_counts, inlier_mask, ws, ws_bytes, stream);
}
