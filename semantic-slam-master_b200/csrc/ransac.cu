// Geometric verification of padded match lists: batched RANSAC for P pairs at once, against a
// homography (HModel) or a fundamental matrix (FModel).  The hypothesis and scoring kernels are
// ransac.cuh's, with the correspondences (x1, y1, x2, y2) staged as float4; the refit is this file's:
//
//   ransac_hyp     one thread per (pair, sample): SAMPLE distinct rows drawn by a counter-based
//                  splitmix64 sampler, minimal solve in double -> SLOTS fp32 hypotheses
//   ransac_score   the hot loop (P x SLOTS*iters x n error evaluations)
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
#include "ransac.cuh"

namespace sslam {
namespace {

constexpr double PIVOT_TOL = 1e-8;    // |pivot| of the normalised 8x8 / 7x9 solves, |h33| before scaling
constexpr int BISECT = 64;            // bisection steps per sign-changing bracket of the 7-point cubic
constexpr double SQRT2 = 1.4142135623730951;

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

// ---------------------------------------------------------------------------- homography model
// The row access of both models: correspondences as float4, staged as float4 (a 64 KB tile, three
// scoring CTAs per SM).
struct CorrRows {
  static constexpr int FLOATS = 9, TILE = 4096, ROW_FLOATS = 4;
  using Row = float4;
  __device__ static float4 row(const RansacParams& r, int p, int a, int b, int k) { return corr(r, p, a, b, k); }
  __device__ static void stage(float* s, int, int k, float4 q) { reinterpret_cast<float4*>(s)[k] = q; }
  __device__ static float4 staged(const float* s, int, int k) { return reinterpret_cast<const float4*>(s)[k]; }
};

// Slots of sample s: bit k of solve()'s result marks slot k valid.  accumulate() adds one inlier's
// normal-matrix terms (upper triangle, 45 sums); finish() turns the smallest eigenvector of the normal
// matrix into the model (thread 0; A, V: 81-double shared scratch).
struct HModel : CorrRows {
  static constexpr int SAMPLE = 4, SLOTS = 1, MIN_FIT = 4;
  __device__ static int solve(const float4 q[SAMPLE], const RansacParams&, double H[SLOTS][FLOATS]) {
    return dlt4(q, H[0]) ? 1 : 0;
  }
  __device__ static bool inlier(const float h[9], float4 q, const RansacParams& r) { return is_inlier(h, q, r.t2); }
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

struct FModel : CorrRows {
  static constexpr int SAMPLE = 7, SLOTS = 3, MIN_FIT = 8;
  __device__ static int solve(const float4 q[SAMPLE], const RansacParams&, double F[SLOTS][FLOATS]) {
    return seven_point(q, F);
  }
  __device__ static bool inlier(const float f[9], float4 q, const RansacParams& r) { return epi_inlier(f, q, r.t2); }
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

// ---------------------------------------------------------------------------- refit
// Hypothesis slot h of pair p as doubles (false: degenerate).
template <class M>
__device__ bool slot_hypothesis(const RansacParams& r, int p, int a, int b, int n, int h, double H[9]) {
  double Hs[M::SLOTS][9];
  const int k = h % M::SLOTS;
  if (!((sample_hyps<M>(r, p, a, b, n, h / M::SLOTS, Hs) >> k) & 1)) return false;
  for (int j = 0; j < 9; ++j) H[j] = Hs[k][j];
  return true;
}

template <class M>
__global__ void __launch_bounds__(GEO_THREADS) ransac_refit_kernel(RansacParams r) {
  __shared__ uint8_t flag[MAX_L];
  __shared__ double red[(GEO_THREADS / 32) * 45];
  __shared__ double sum[45];
  __shared__ double Aj[81], Vj[81];
  __shared__ double Hs[2][9];                       // [0] best hypothesis, [1] refit
  __shared__ float hf[9];
  __shared__ int scan[GEO_THREADS];
  __shared__ unsigned long long bkey[GEO_THREADS / 32];
  __shared__ int s_best, s_ok, s_total;
  const int p = blockIdx.x, tid = threadIdx.x;
  int a, b;
  const int n = pair_rows(r, p, a, b);

  // ---- best hypothesis
  best_keys<M>(r, p, n, bkey);
  if (tid == 0) {
    const int best = best_slot(bkey);
    s_ok = best >= 0 && slot_hypothesis<M>(r, p, a, b, n, best, Hs[0]);
    s_best = s_ok ? best : -1;
    if (s_ok)
      for (int k2 = 0; k2 < 9; ++k2) hf[k2] = __double2float_rn(Hs[0][k2]);
  }
  __syncthreads();
  const bool have = s_ok;
  const int m = mask_pass<M>(r, p, a, b, n, have, hf, flag, scan);

  // ---- refit over the best hypothesis's inliers (normalised least squares)
  bool use_refit = false;
  if (have && m >= M::MIN_FIT) {
    double c4[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k = tid; k < n; k += GEO_THREADS)
      if (flag[k]) {
        const float4 q = corr(r, p, a, b, k);
        c4[0] = dadd(c4[0], q.x); c4[1] = dadd(c4[1], q.y); c4[2] = dadd(c4[2], q.z); c4[3] = dadd(c4[3], q.w);
      }
    block_sum<4>(c4, red, sum);
    const double cx1 = sum[0] / m, cy1 = sum[1] / m, cx2 = sum[2] / m, cy2 = sum[3] / m;
    double d2[2] = {0.0, 0.0};
    for (int k = tid; k < n; k += GEO_THREADS)
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
      for (int k = tid; k < n; k += GEO_THREADS)
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
      if (s_ok) use_refit = keep_refit<M>(r, p, a, b, n, hf, m, scan);
    }
  }
  __syncthreads();
  if (use_refit)
    for (int k = tid; k < n; k += GEO_THREADS) flag[k] = M::inlier(hf, M::row(r, p, a, b, k), r);
  if (tid == 0) r.best[p] = s_best;
  if (r.H && tid < 9) r.H[9 * (size_t)p + tid] = have ? Hs[use_refit ? 1 : 0][tid] : 0.0;
  finish_lists(r, p, n, flag, scan, &s_total);
}

template <class Model>
int ransac(const float* kpts1, int F1, const float* kpts2, int F2, const int32_t* pair_index, int P, int N, int M,
           const int32_t* pairs, const float* pair_scores, const int32_t* counts, int L, int iters, double threshold,
           uint64_t seed, double* H, int32_t* out_pairs, float* out_scores, int32_t* out_counts,
           uint8_t* inlier_mask, void* ws, size_t ws_bytes, void* stream) {
  int rc = check_device();
  if (rc) return rc;
  rc = check_list_args("ransac", P, N, M, L, F1, F2, pair_index,
                       kpts1 && kpts2 && pairs && pair_scores && counts && out_pairs && out_scores && out_counts && ws,
                       &iters, nullptr, "threshold", threshold, nullptr);
  if (rc || P == 0) return rc;
  RansacParams r{kpts1, kpts2, F1, F2, pair_index, P, N, M, pairs, pair_scores, counts, L, iters,
                 (float)(threshold * threshold), (u64)seed, H, out_pairs, out_scores, out_counts, inlier_mask};
  return ransac_launch<Model>("ransac", r, ws, ws_bytes, ransac_refit_kernel<Model>,
                              {KK_RANSAC_HYP, KK_RANSAC_SCORE, KK_RANSAC_REFIT}, (cudaStream_t)stream);
}

}  // namespace
}  // namespace sslam

using namespace sslam;

extern "C" size_t sslam_ransac_workspace_bytes(int P, int L, int iters) {
  return ransac_workspace_bytes<HModel>(P, L, iters);
}

extern "C" size_t sslam_ransac_fundamental_workspace_bytes(int P, int L, int iters) {
  return ransac_workspace_bytes<FModel>(P, L, iters);
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
