// Camera tracking from 2D-3D match lists: batched P3P RANSAC for P lists at once, three launches.  The
// hypothesis and scoring kernels are ransac.cuh's, ransac_hyp<PModel> and ransac_score<PModel>; the refit
// is this file's.
//
//   pnp_hyp    one thread per (list, sample): 4 distinct rows by the splitmix64 sampler; rows 0-2 go to
//              the Lambda Twist P3P solver (Persson & Nordberg, ECCV 2018) in double, row 3 picks among
//              its up to 4 solutions (least squared reprojection error, lowest solution on ties) ->
//              one fp32 hypothesis (R, t) per sample
//   pnp_score  the hot loop (P x iters x n reprojection tests): the list's rows (X, Y, Z, u, v) are staged
//              in shared memory tile by tile as five float arrays, warps take hypotheses, lanes stride rows
//   pnp_refit  one CTA per list: best sample (most inliers, lowest sample on ties), Levenberg-Marquardt in
//              6 DOF on the reprojection error of its inliers (one block_sum<28> per relinearisation),
//              re-score, order-preserving compaction into the matcher's list format
//
// Every result is a function of (inputs, iters, threshold, seed, refine_iters) only, and no reduction uses
// atomics.  The hypothesis path uses correctly rounded operations only (__dmul_rn / __dadd_rn / __ddiv_rn
// / __dsqrt_rn, __fmul_rn / __fadd_rn / __frcp_rn) in fixed orders with fixed iteration counts; oracle/pnp.py
// restates it operation by operation, so counts, best sample and pre-refit mask agree bit for bit.
#include "ransac.cuh"

namespace sslam {
namespace {

constexpr int HF = 12;                // floats per hypothesis: R row-major (9), t (3)
constexpr int CUBIC_BISECT = 100;     // bisection steps for the root of the P3P cubic
constexpr int GN_STEPS = 5;           // Gauss-Newton steps on the P3P depths
constexpr double COLLINEAR_TOL = 1e-12;   // |d12 x d13|^2 <= tol |d12|^2 |d13|^2: collinear or coincident
constexpr int MIN_REFINE_ROWS = 4;
constexpr int NP = 6;                 // refinement parameters: w (3), d (3)
constexpr int NJ = lm_nj(NP);

struct PnpRow { float X, Y, Z, u, v; };

// Row k as X, Y, Z (the 3-D point) and u, v (the keypoint); NaN (never an inlier, degenerate sample) when
// an index is out of range.
__device__ __forceinline__ PnpRow pnp_row(const RansacParams& r, int p, int a, int b, int k) {
  const int2 ij = reinterpret_cast<const int2*>(r.pairs)[(size_t)p * r.L + k];
  if (ij.x < 0 || ij.x >= r.N || ij.y < 0 || ij.y >= r.M) {
    const float nan = __int_as_float(0x7fc00000);
    return {nan, nan, nan, nan, nan};
  }
  const float* X = r.k1 + ((size_t)a * r.N + ij.x) * 3;
  const float2 v = reinterpret_cast<const float2*>(r.k2)[(size_t)b * r.M + ij.y];
  return {X[0], X[1], X[2], v.x, v.y};
}

// Roots of x^2 + b x + c (Lambda Twist's root2real, a negative discriminant clamped to 0).
__device__ __forceinline__ void root2(double b, double c, double& r1, double& r2) {
  const double v = dsub(dmul(b, b), dmul(4.0, c));
  const double y = __dsqrt_rn(v > 0.0 ? v : 0.0);
  if (b < 0.0) {
    const double s = dadd(-b, y);
    r1 = dmul(0.5, s);
    r2 = __ddiv_rn(dmul(2.0, c), s);
  } else {
    const double s = dsub(-b, y);
    r1 = __ddiv_rn(dmul(2.0, c), s);
    r2 = dmul(0.5, s);
  }
}

// Eigenvector of the symmetric A (a00, a01, a02, a11, a12, a22) for eigenvalue e, from its first two rows
// with the last component set to 1, then normalised (Lambda Twist's eigwithknown0).
__device__ __forceinline__ void eigvec(const double A[6], double e, double mx0011, double x01sq, double prec0,
                                       double prec1, double v[3]) {
  const double den = dadd(dsub(dadd(dmul(e, dadd(A[0], A[3])), mx0011), dmul(e, e)), x01sq);
  const double tmp = __ddiv_rn(1.0, den);
  const double a1 = dmul(-dadd(dmul(e, A[2]), prec0), tmp);
  const double a2 = dmul(-dadd(dmul(e, A[4]), prec1), tmp);
  const double rn = __ddiv_rn(1.0, __dsqrt_rn(dadd(dadd(dmul(a1, a1), dmul(a2, a2)), 1.0)));
  v[0] = dmul(a1, rn); v[1] = dmul(a2, rn); v[2] = rn;
}

__device__ __forceinline__ double gn_cost(const double l[3], double a12, double a13, double a23, double b12,
                                          double b13, double b23, double res[3]) {
  res[0] = dsub(dadd(dadd(dmul(l[0], l[0]), dmul(l[1], l[1])), dmul(dmul(b12, l[0]), l[1])), a12);
  res[1] = dsub(dadd(dadd(dmul(l[0], l[0]), dmul(l[2], l[2])), dmul(dmul(b13, l[0]), l[2])), a13);
  res[2] = dsub(dadd(dadd(dmul(l[1], l[1]), dmul(l[2], l[2])), dmul(dmul(b23, l[1]), l[2])), a23);
  return dadd(dadd(fabs(res[0]), fabs(res[1])), fabs(res[2]));
}

// GN_STEPS Gauss-Newton steps on the depths l (Lambda Twist's gauss_newton_refineL): stop when the
// residual's 1-norm is below 1e-10, reject (and stop at) a step that increases it.
__device__ __forceinline__ void refine_depths(double l[3], double a12, double a13, double a23, double b12,
                                              double b13, double b23) {
  for (int it = 0; it < GN_STEPS; ++it) {
    double res[3], rn[3];
    const double c0 = gn_cost(l, a12, a13, a23, b12, b13, b23, res);
    if (c0 < 1e-10) break;
    const double v0 = dadd(dmul(2.0, l[0]), dmul(b12, l[1])), v1 = dadd(dmul(2.0, l[1]), dmul(b12, l[0]));
    const double v3 = dadd(dmul(2.0, l[0]), dmul(b13, l[2])), v5 = dadd(dmul(2.0, l[2]), dmul(b13, l[0]));
    const double v7 = dadd(dmul(2.0, l[1]), dmul(b23, l[2])), v8 = dadd(dmul(2.0, l[2]), dmul(b23, l[1]));
    const double det = __ddiv_rn(1.0, dsub(dmul(dmul(-v0, v5), v7), dmul(dmul(v1, v3), v8)));
    const double j0 = dadd(dadd(dmul(dmul(-v5, v7), res[0]), dmul(dmul(-v1, v8), res[1])), dmul(dmul(v1, v5), res[2]));
    const double j1 = dadd(dadd(dmul(dmul(-v3, v8), res[0]), dmul(dmul(v0, v8), res[1])), dmul(dmul(-v0, v5), res[2]));
    const double j2 = dadd(dadd(dmul(dmul(v3, v7), res[0]), dmul(dmul(-v0, v7), res[1])), dmul(dmul(-v1, v3), res[2]));
    const double ln[3] = {dsub(l[0], dmul(det, j0)), dsub(l[1], dmul(det, j1)), dsub(l[2], dmul(det, j2))};
    if (gn_cost(ln, a12, a13, a23, b12, b13, b23, rn) > c0) break;
    l[0] = ln[0]; l[1] = ln[1]; l[2] = ln[2];
  }
}

// Lambda Twist P3P: bearings y[3] (unit), world points x[3] -> up to 4 poses (x_cam = R x + t) in Rs, ts.
// Returns the number of solutions; 0 when the points are collinear or coincident (COLLINEAR_TOL), the
// cubic is degenerate, or no real solution with positive depths exists.  The cubic's root: the Cauchy
// bound B = 1 + max |k_i| brackets a real root of the monic x^3 + k2 x^2 + k1 x + k0 in [-B, B], bisected
// CUBIC_BISECT times.  Not inlined: it is the bulk of pnp_hyp and, on thread 0, of pnp_refit.
__device__ __noinline__ int p3p(const double y[3][3], const double x[3][3], double Rs[4][9], double ts[4][3]) {
  const double b12 = dmul(-2.0, dot3(y[0], y[1])), b13 = dmul(-2.0, dot3(y[0], y[2]));
  const double b23 = dmul(-2.0, dot3(y[1], y[2]));
  double d12[3], d13[3], d23[3], c[3];
  for (int i = 0; i < 3; ++i) {
    d12[i] = dsub(x[0][i], x[1][i]); d13[i] = dsub(x[0][i], x[2][i]); d23[i] = dsub(x[1][i], x[2][i]);
  }
  cross3(d12, d13, c);
  const double a12 = dot3(d12, d12), a13 = dot3(d13, d13), a23 = dot3(d23, d23);
  const double cc = dot3(c, c);
  if (!(cc > dmul(dmul(COLLINEAR_TOL, a12), a13))) return 0;
  const double c31 = dmul(-0.5, b13), c23 = dmul(-0.5, b23), c12 = dmul(-0.5, b12);
  const double blob = dsub(dmul(dmul(c12, c23), c31), 1.0);
  const double s31 = dsub(1.0, dmul(c31, c31)), s23 = dsub(1.0, dmul(c23, c23)), s12 = dsub(1.0, dmul(c12, c12));
  const double p3 = dmul(a13, dsub(dmul(a23, s31), dmul(a13, s23)));
  const double p2 = dadd(dadd(dmul(dmul(dmul(2.0, blob), a23), a13), dmul(dmul(a13, dadd(dmul(2.0, a12), a13)), s23)),
                         dmul(dmul(a23, dsub(a23, a12)), s31));
  const double p1 = dsub(dsub(dmul(dmul(a23, dsub(a13, a23)), s12), dmul(dmul(a12, a12), s23)),
                         dmul(dmul(2.0, a12), dadd(dmul(blob, a23), dmul(a13, s23))));
  const double p0 = dmul(a12, dsub(dmul(a12, s23), dmul(a23, s12)));
  if (!(p3 != 0.0) || !isfinite(p3)) return 0;
  const double k2 = __ddiv_rn(p2, p3), k1 = __ddiv_rn(p1, p3), k0 = __ddiv_rn(p0, p3);
  const double B = dadd(1.0, fmax(fmax(fabs(k2), fabs(k1)), fabs(k0)));
  if (!isfinite(B)) return 0;
  double lo = -B, hi = B;
  for (int it = 0; it < CUBIC_BISECT; ++it) {
    const double m = dmul(dadd(lo, hi), 0.5);
    const double f = dadd(dmul(dadd(dmul(dadd(m, k2), m), k1), m), k0);
    if (f < 0.0) lo = m; else hi = m;
  }
  const double g = dmul(dadd(lo, hi), 0.5);
  // A = D1 + g D2, rank 2
  double A[6];
  A[0] = dmul(a23, dsub(1.0, g));
  A[1] = dmul(dmul(a23, b12), 0.5);
  A[2] = dmul(dmul(dmul(a23, b13), g), -0.5);
  A[3] = dadd(dsub(a23, a12), dmul(a13, g));
  A[4] = dmul(dmul(b23, dsub(dmul(a13, g), a12)), 0.5);
  A[5] = dsub(dmul(g, dsub(a13, a23)), a12);
  const double x01sq = dmul(A[1], A[1]);
  const double eb = dsub(dsub(-A[0], A[3]), A[5]);
  const double ec = dadd(dadd(dsub(dsub(-x01sq, dmul(A[2], A[2])), dmul(A[4], A[4])), dmul(A[0], dadd(A[3], A[5]))),
                         dmul(A[3], A[5]));
  double e1, e2;
  root2(eb, ec, e1, e2);
  if (fabs(e1) < fabs(e2)) { const double s = e1; e1 = e2; e2 = s; }
  const double mx0011 = dmul(-A[0], A[3]);
  const double prec0 = dsub(dmul(A[1], A[4]), dmul(A[2], A[3]));
  const double prec1 = dsub(dmul(A[1], A[2]), dmul(A[0], A[4]));
  double v1[3], v2[3];
  eigvec(A, e1, mx0011, x01sq, prec0, prec1, v1);
  eigvec(A, e2, mx0011, x01sq, prec0, prec1, v2);
  const double q = -__ddiv_rn(e2, e1);
  const double sv = __dsqrt_rn(q > 0.0 ? q : 0.0);
  double Ls[4][3];
  int nsol = 0;
  for (int sgn = 0; sgn < 2; ++sgn) {
    const double s = sgn == 0 ? sv : -sv;
    const double w2 = __ddiv_rn(1.0, dsub(dmul(s, v2[0]), v1[0]));
    const double w0 = dmul(dsub(v1[1], dmul(s, v2[1])), w2);
    const double w1 = dmul(dsub(v1[2], dmul(s, v2[2])), w2);
    const double a = __ddiv_rn(1.0, dsub(dsub(dmul(dmul(dsub(a13, a12), w1), w1), dmul(dmul(a12, b13), w1)), a12));
    const double bb = dmul(dsub(dsub(dmul(dmul(a13, b12), w1), dmul(dmul(a12, b13), w0)),
                                dmul(dmul(dmul(2.0, w0), w1), dsub(a12, a13))), a);
    const double cq = dmul(dadd(dadd(dmul(dmul(dsub(a13, a12), w0), w0), dmul(dmul(a13, b12), w0)), a13), a);
    if (!(dsub(dmul(bb, bb), dmul(4.0, cq)) >= 0.0)) continue;
    double tau[2];
    root2(bb, cq, tau[0], tau[1]);
    for (int k = 0; k < 2; ++k) {
      if (!(tau[k] > 0.0)) continue;
      const double d = __ddiv_rn(a23, dadd(dmul(tau[k], dadd(b23, tau[k])), 1.0));
      if (!(d > 0.0)) continue;
      const double l2 = __dsqrt_rn(d), l3 = dmul(tau[k], l2);
      const double l1 = dadd(dmul(w0, l2), dmul(w1, l3));
      if (!(l1 >= 0.0)) continue;
      Ls[nsol][0] = l1; Ls[nsol][1] = l2; Ls[nsol][2] = l3;
      ++nsol;
    }
  }
  // X^-1 of the columns [d12, d13, c]: rows (d13 x c, c x d12, d12 x d13) / det, det = c.c
  double Xi[3][3];
  cross3(d13, c, Xi[0]);
  cross3(c, d12, Xi[1]);
  for (int i = 0; i < 3; ++i) {
    Xi[0][i] = __ddiv_rn(Xi[0][i], cc); Xi[1][i] = __ddiv_rn(Xi[1][i], cc); Xi[2][i] = __ddiv_rn(c[i], cc);
  }
  for (int i = 0; i < nsol; ++i) {
    refine_depths(Ls[i], a12, a13, a23, b12, b13, b23);
    double ry[3][3], yd1[3], yd2[3], yc[3];
    for (int k = 0; k < 3; ++k)
      for (int j = 0; j < 3; ++j) ry[k][j] = dmul(y[k][j], Ls[i][k]);
    for (int j = 0; j < 3; ++j) { yd1[j] = dsub(ry[0][j], ry[1][j]); yd2[j] = dsub(ry[0][j], ry[2][j]); }
    cross3(yd1, yd2, yc);
    for (int r = 0; r < 3; ++r)
      for (int j = 0; j < 3; ++j)
        Rs[i][3 * r + j] = dadd(dadd(dmul(yd1[r], Xi[0][j]), dmul(yd2[r], Xi[1][j])), dmul(yc[r], Xi[2][j]));
    for (int r = 0; r < 3; ++r) ts[i][r] = dsub(ry[0][r], dot3(Rs[i] + 3 * r, x[0]));
  }
  return nsol;
}

// Pose (R row-major, t) of the sample's rows q (false: degenerate).  Rows 0-2 go to p3p; among its
// solutions that are finite and put all four points at z > 0, row 3 picks the one with the least squared
// reprojection error (fx Xc / Zc + cx - u)^2 + (fy Yc / Zc + cy - v)^2, the lowest solution on ties.
__device__ bool sample_pose(const PnpRow q[4], const RansacParams& r, double H[HF]) {
  double X[4][3], uv[4][2];
  bool fin = true;
  for (int k = 0; k < 4; ++k) {
    fin &= isfinite(q[k].X) & isfinite(q[k].Y) & isfinite(q[k].Z) & isfinite(q[k].u) & isfinite(q[k].v);
    X[k][0] = q[k].X; X[k][1] = q[k].Y; X[k][2] = q[k].Z; uv[k][0] = q[k].u; uv[k][1] = q[k].v;
  }
  if (!fin) return false;
  double y[3][3];
  for (int k = 0; k < 3; ++k) {
    const double f0 = __ddiv_rn(dsub(uv[k][0], r.cx), r.fx), f1 = __ddiv_rn(dsub(uv[k][1], r.cy), r.fy);
    const double nrm = __dsqrt_rn(dadd(dadd(dmul(f0, f0), dmul(f1, f1)), 1.0));
    y[k][0] = __ddiv_rn(f0, nrm); y[k][1] = __ddiv_rn(f1, nrm); y[k][2] = __ddiv_rn(1.0, nrm);
  }
  double Rs[4][9], ts[4][3];
  const int ns = p3p(y, X, Rs, ts);
  int best = -1;
  double be = 0.0;
  for (int i = 0; i < ns; ++i) {
    bool ok = true;
    for (int j = 0; j < 9; ++j) ok &= isfinite(Rs[i][j]);
    for (int j = 0; j < 3; ++j) ok &= isfinite(ts[i][j]);
    for (int k = 0; k < 4; ++k) ok &= dadd(dot3(Rs[i] + 6, X[k]), ts[i][2]) > 0.0;
    if (!ok) continue;
    const double xc = dadd(dot3(Rs[i], X[3]), ts[i][0]), yc = dadd(dot3(Rs[i] + 3, X[3]), ts[i][1]);
    const double zc = dadd(dot3(Rs[i] + 6, X[3]), ts[i][2]);
    const double du = dsub(dadd(dmul(r.fx, __ddiv_rn(xc, zc)), r.cx), uv[3][0]);
    const double dv = dsub(dadd(dmul(r.fy, __ddiv_rn(yc, zc)), r.cy), uv[3][1]);
    const double e = dadd(dmul(du, du), dmul(dv, dv));
    if (best < 0 || e < be) { best = i; be = e; }
  }
  if (best < 0) return false;
  for (int j = 0; j < 9; ++j) H[j] = Rs[best][j];
  for (int j = 0; j < 3; ++j) H[9 + j] = ts[best][j];
  return true;
}

// Inlier test in fp32, no contraction: Xc = ((R0 X + R1 Y) + R2 Z) + t0 (likewise Yc, Zc), iz = rcp(Zc),
// du = (fx Xc) iz + cx - u, dv = (fy Yc) iz + cy - v; inlier iff Zc > 0 and du du + dv dv < t2.
__device__ __forceinline__ bool pnp_inlier(const float h[HF], const PnpRow& q, const RansacParams& r) {
  const float fx = (float)r.fx, fy = (float)r.fy, cx = (float)r.cx, cy = (float)r.cy;
  const float xc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[0], q.X), __fmul_rn(h[1], q.Y)), __fmul_rn(h[2], q.Z)), h[9]);
  const float yc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[3], q.X), __fmul_rn(h[4], q.Y)), __fmul_rn(h[5], q.Z)), h[10]);
  const float zc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[6], q.X), __fmul_rn(h[7], q.Y)), __fmul_rn(h[8], q.Z)), h[11]);
  const float iz = __frcp_rn(zc);
  const float du = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(fx, xc), iz), cx), q.u);
  const float dv = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(fy, yc), iz), cy), q.v);
  return zc > 0.f && __fadd_rn(__fmul_rn(du, du), __fmul_rn(dv, dv)) < r.t2;
}

// The PnP model of ransac.cuh: 4-row samples, one pose per sample; rows staged as five float arrays
// (X, Y, Z, u, v): 60 KB at 3072 rows plus 13 KB static, three scoring CTAs per SM.
struct PModel {
  static constexpr int SAMPLE = 4, SLOTS = 1, FLOATS = HF, TILE = 3072, ROW_FLOATS = 5;
  using Row = PnpRow;
  __device__ static PnpRow row(const RansacParams& r, int p, int a, int b, int k) { return pnp_row(r, p, a, b, k); }
  __device__ static void stage(float* s, int tile, int k, const PnpRow& q) {
    s[k] = q.X; s[tile + k] = q.Y; s[2 * tile + k] = q.Z; s[3 * tile + k] = q.u; s[4 * tile + k] = q.v;
  }
  __device__ static PnpRow staged(const float* s, int tile, int k) {
    return {s[k], s[tile + k], s[2 * tile + k], s[3 * tile + k], s[4 * tile + k]};
  }
  __device__ static bool inlier(const float h[HF], const PnpRow& q, const RansacParams& r) { return pnp_inlier(h, q, r); }
  __device__ static int solve(const PnpRow q[SAMPLE], const RansacParams& r, double H[SLOTS][HF]) {
    return sample_pose(q, r, H[0]) ? 1 : 0;
  }
};

// Reprojection residual (px) of one row under H = (R, t) in double, and optionally its Jacobian along
// (w, d) for R <- Exp(w) R, t <- t + d: dXc/dw_j = e_j x (R X), dXc/dd = I.
__device__ __forceinline__ void reproj(const double* H, const PnpRow& q, double fx, double fy, double cx,
                                       double cy, double res[2], double (*J)[NP]) {
  const double* R = H;
  const double* t = H + 9;
  const double X[3] = {q.X, q.Y, q.Z};
  const double rx[3] = {dot3(R, X), dot3(R + 3, X), dot3(R + 6, X)};
  const double xc = dadd(rx[0], t[0]), yc = dadd(rx[1], t[1]), zc = dadd(rx[2], t[2]);
  const double iz = __ddiv_rn(1.0, zc);
  const double pu = dmul(xc, iz), pv = dmul(yc, iz);
  res[0] = dsub(dadd(dmul(fx, pu), cx), (double)q.u);
  res[1] = dsub(dadd(dmul(fy, pv), cy), (double)q.v);
  if (!J) return;
  const double gu[3] = {dmul(fx, iz), 0.0, -dmul(dmul(fx, pu), iz)};
  const double gv[3] = {0.0, dmul(fy, iz), -dmul(dmul(fy, pv), iz)};
  const double col[3][3] = {{0.0, -rx[2], rx[1]}, {rx[2], 0.0, -rx[0]}, {-rx[1], rx[0], 0.0}};
  for (int j = 0; j < 3; ++j) {
    J[0][j] = dot3(gu, col[j]);
    J[1][j] = dot3(gv, col[j]);
    J[0][3 + j] = gu[j];
    J[1][3 + j] = gv[j];
  }
}

// One LM trial (thread 0): the damped step x, candidate Rn = Exp(x_w) R, tn = t + x_d (Hn = (Rn, tn)).
// false: no step.
__device__ __noinline__ bool lm_step(const double* Js, double lam, const double* H, double* Hn) {
  double x[NP];
  if (!lm_solve<NP>(Js, lam, x)) return false;
  double X[9];
  rodrigues(x, X);
  mat3(X, H, Hn);
  for (int i = 0; i < 3; ++i) Hn[9 + i] = dadd(H[9 + i], x[3 + i]);
  return true;
}

// Best sample of list p into H[0] on thread 0 (false: none); not inlined, so that the P3P solve stays out
// of the row loops' registers.
__device__ __noinline__ bool best_pose(const RansacParams& r, int p, int a, int b, int n, int best, double (*H)[HF]) {
  return best >= 0 && sample_hyps<PModel>(r, p, a, b, n, best, H) != 0;
}

// One CTA per SM (minBlocksPerSM = 1): under the two-CTA register cap of 128, ptxas spills in p3p and
// best_pose on thread 0's path.
__global__ void __launch_bounds__(GEO_THREADS, 1) pnp_refit_kernel(RansacParams r) {
  __shared__ uint8_t flag[MAX_L];
  __shared__ double red[(GEO_THREADS / 32) * NJ];
  __shared__ double sum[NJ];
  __shared__ double sH[2][HF], nH[HF];                // [0] best sample, [1] refined; LM candidate
  __shared__ float hf[HF];
  __shared__ int scan[GEO_THREADS];
  __shared__ unsigned long long bkey[GEO_THREADS / 32];
  __shared__ int s_best, s_ok, s_total;
  const int p = blockIdx.x, tid = threadIdx.x;
  int a, b;
  const int n = pair_rows(r, p, a, b);
  const double fx = r.fx, fy = r.fy, cx = r.cx, cy = r.cy;

  // ---- best sample
  best_keys<PModel>(r, p, n, bkey);
  if (tid == 0) {
    const int best = best_slot(bkey);
    s_ok = best_pose(r, p, a, b, n, best, sH);
    s_best = s_ok ? best : -1;
    if (s_ok)
      for (int k2 = 0; k2 < HF; ++k2) hf[k2] = __double2float_rn(sH[0][k2]);
  }
  __syncthreads();
  const bool have = s_ok;
  const int m = mask_pass<PModel>(r, p, a, b, n, have, hf, flag, scan);

  // ---- Levenberg-Marquardt over the best sample's inliers
  double2 cost = make_double2(0.0, 0.0);              // r^T r before / after
  bool use_refit = false;
  if (have && m > 0) {
    if (tid < HF) sH[1][tid] = sH[0][tid];
    __syncthreads();
    const bool refine = r.refine_iters > 0 && m >= MIN_REFINE_ROWS;
    auto acc_row = [&](int k, double (&acc)[NJ]) {
      if (!flag[k]) return;
      double res[2], J[2][NP];
      reproj(sH[1], pnp_row(r, p, a, b, k), fx, fy, cx, cy, res, J);
#pragma unroll
      for (int e = 0; e < 2; ++e) lm_add<NP>(acc, J[e], res[e]);
    };
    auto cost_row = [&](int k, double& c) {
      if (!flag[k]) return;
      double res[2];
      reproj(nH, pnp_row(r, p, a, b, k), fx, fy, cx, cy, res, nullptr);
      c = dadd(c, dadd(dmul(res[0], res[0]), dmul(res[1], res[1])));
    };
    auto step = [&](const double* J, double lam) { return lm_step(J, lam, sH[1], nH); };
    auto commit = [&] {
      for (int i = 0; i < HF; ++i) sH[1][i] = nH[i];
    };
    cost = lm_refine<NP>(n, refine, r.refine_iters, red, sum, acc_row, cost_row, step, commit);
    // ---- re-score with the refined pose: kept iff it has at least as many inliers
    if (refine) {
      if (tid == 0)
        for (int k2 = 0; k2 < HF; ++k2) hf[k2] = __double2float_rn(sH[1][k2]);
      __syncthreads();
      use_refit = keep_refit<PModel>(r, p, a, b, n, hf, m, scan);
    }
  }
  __syncthreads();
  if (use_refit)
    for (int k = tid; k < n; k += GEO_THREADS) flag[k] = pnp_inlier(hf, pnp_row(r, p, a, b, k), r);
  if (tid == 0) r.best[p] = s_best;
  const int sel = use_refit ? 1 : 0;
  const bool model = have && m > 0;                   // a best sample without an inlier is no model
  if (tid < 9) r.R[9 * (size_t)p + tid] = model ? sH[sel][tid] : 0.0;
  if (tid < 3) r.t[3 * (size_t)p + tid] = model ? sH[sel][9 + tid] : 0.0;
  if (r.rms && tid < 2) {
    const double c = tid == 0 || !use_refit ? cost.x : cost.y;
    r.rms[2 * (size_t)p + tid] = model ? __dsqrt_rn(__ddiv_rn(c, (double)m)) : 0.0;
  }
  finish_lists(r, p, n, flag, scan, &s_total);
}

}  // namespace
}  // namespace sslam

using namespace sslam;

extern "C" size_t sslam_ransac_pnp_workspace_bytes(int P, int L, int iters) {
  return ransac_workspace_bytes<PModel>(P, L, iters);
}

extern "C" int sslam_ransac_pnp(const float* points, int F1, const float* kpts2, int F2, const int32_t* pair_index,
                                int P, int N, int M, const int32_t* pairs, const float* pair_scores,
                                const int32_t* counts, int L, double fx, double fy, double cx, double cy, int iters,
                                double threshold, uint64_t seed, int refine_iters, double* R, double* t,
                                double* rms, int32_t* out_pairs, float* out_scores, int32_t* out_counts,
                                uint8_t* inlier_mask, void* ws, size_t ws_bytes, void* stream) {
  int rc = check_device();
  if (rc) return rc;
  const double K[4] = {fx, fy, cx, cy};
  rc = check_list_args("ransac_pnp", P, N, M, L, F1, F2, pair_index,
                       points && kpts2 && pairs && pair_scores && counts && R && t && out_pairs && out_scores &&
                           out_counts && ws,
                       &iters, &refine_iters, "threshold", threshold, K);
  if (rc || P == 0) return rc;
  RansacParams r{points, kpts2, F1, F2, pair_index, P, N, M, pairs, pair_scores, counts, L, iters,
                 (float)(threshold * threshold), (u64)seed, nullptr, out_pairs, out_scores, out_counts, inlier_mask,
                 nullptr, nullptr, nullptr, nullptr, fx, fy, cx, cy, refine_iters, R, t, rms};
  return ransac_launch<PModel>("ransac_pnp", r, ws, ws_bytes, pnp_refit_kernel,
                               {KK_PNP_HYP, KK_PNP_SCORE, KK_PNP_REFIT}, (cudaStream_t)stream);
}
