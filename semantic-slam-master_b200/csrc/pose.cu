// Relative pose from verified match lists: one CTA (256 threads) per pair, one launch, no workspace.
//
//   decomposition  thread 0, double: E / |E|_F, eigenvectors of E^T E by Jacobi (descending eigenvalue,
//                  lowest index on ties, v3 negated when det V < 0), U by Gram-Schmidt on E v1, E v2,
//                  u3 = u1 x u2; with cv2's W, R_a = U W V^T, R_b = U W^T V^T, t = u3; candidates
//                  (R_a, t), (R_b, t), (R_a, -t), (R_b, -t)
//   cheirality    one thread per row, double, correctly rounded operations: midpoint depths of the rays
//                  f1 = K^-1 x1 (rotated: u = R f1) and f2 = K^-1 x2; a row is good iff the rays are not
//                  parallel and the point lies in front of both cameras closer than distance_thresh
//                  (cv2.recoverPose's rule); the candidate with the most good rows wins (lowest on ties)
//   refinement     Levenberg-Marquardt on (R, t) in 5 DOF — R <- Exp(w) R, t <- normalise(t + d1 b1 + d2 b2)
//                  — over the signed Sampson distance in pixels of every usable row; J^T J, J^T r and r^T r
//                  in one fixed-order block reduction per relinearisation, the 5x5 damped solve on thread 0
//   final pass     cheirality with the refined pose: mask, points, order-preserving compaction of the good
//                  rows into the matcher's list format
//
// Every result is a function of the pair's own inputs: no reduction uses atomics and nothing depends on
// the pair's position in the batch.  oracle/pose.py restates every stage in NumPy float64.
#include "geometry.cuh"

namespace sslam {
namespace {

constexpr int MIN_REFINE_ROWS = 5;    // rows the 5-DOF refinement needs
constexpr int NP = 5;                 // refinement parameters: w (3), d (2)
constexpr int NJ = lm_nj(NP);

struct PoseParams {
  const float* k1; const float* k2;          // [F1,N,2], [F2,M,2]
  int F1, F2;
  const int32_t* pair_index;                 // [P,2] or null
  int P, N, M;
  const double* E;                           // [P,9]
  const int32_t* pairs; const float* pair_scores; const int32_t* counts;   // [P,L,2], [P,L], [P]
  int L;
  double fx, fy, cx, cy, dist;
  int iters;
  double* R; double* t;                      // [P,9], [P,3]
  int32_t* cand_good;                        // [P,4] or null
  double* rms;                               // [P,2] or null
  float* points;                             // [P,L,3] or null
  int32_t* out_pairs; float* out_scores; int32_t* out_counts; uint8_t* mask;
};

// f2^T E f1, and the first two entries of F x1 = K^-T E f1 and F^T x2 = K^-T E^T f2 (pixel units).
__device__ __forceinline__ double epi_terms(const double* E, const double f1[3], const double f2[3], double fx,
                                            double fy, double l[4]) {
  const double g0 = dot3(E, f1), g1 = dot3(E + 3, f1), g2 = dot3(E + 6, f1);
  const double h0 = dadd(dadd(dmul(E[0], f2[0]), dmul(E[3], f2[1])), dmul(E[6], f2[2]));
  const double h1 = dadd(dadd(dmul(E[1], f2[0]), dmul(E[4], f2[1])), dmul(E[7], f2[2]));
  l[0] = __ddiv_rn(g0, fx); l[1] = __ddiv_rn(g1, fy); l[2] = __ddiv_rn(h0, fx); l[3] = __ddiv_rn(h1, fy);
  const double g[3] = {g0, g1, g2};
  return dot3(f2, g);
}

__device__ __forceinline__ double dot4(const double* a, const double* b) {
  return dadd(dadd(dadd(dmul(a[0], b[0]), dmul(a[1], b[1])), dmul(a[2], b[2])), dmul(a[3], b[3]));
}

// Signed Sampson distance in pixels, x2^T F x1 / sqrt((F x1)_0^2 + (F x1)_1^2 + (F^T x2)_0^2 + (F^T x2)_1^2),
// 0 when the denominator is 0; s: the square root (0 then).
__device__ __forceinline__ double sampson(const double* E, const double f1[3], const double f2[3], double fx,
                                          double fy, double l[4], double& s) {
  const double num = epi_terms(E, f1, f2, fx, fy, l);
  const double s2 = dot4(l, l);
  s = __dsqrt_rn(s2);
  return s2 > 0.0 ? __ddiv_rn(num, s) : 0.0;
}

// v / |v|; false when |v| is 0 or not finite.
__device__ __forceinline__ bool normalise3(double* v) {
  const double nrm = __dsqrt_rn(dot3(v, v));
  if (!(nrm > 0.0) || !isfinite(nrm)) return false;
  for (int i = 0; i < 3; ++i) v[i] = __ddiv_rn(v[i], nrm);
  return true;
}

// The four candidates of E (thread 0): Rc[0] = R_a, Rc[1] = R_b, t = u3.  false: E is zero, not finite,
// or of rank < 2 (sigma2 <= 1e-12 sigma1).  Not inlined: it keeps the Jacobi out of the row loops' registers.
__device__ __noinline__ bool decompose(const double* Ein, double Rc[2][9], double t[3]) {
  double e[9];
  double n2 = 0.0;
  for (int k = 0; k < 9; ++k) { e[k] = Ein[k]; n2 = dadd(n2, dmul(e[k], e[k])); }
  const double nrm = __dsqrt_rn(n2);
  if (!(nrm > 0.0) || !isfinite(nrm)) return false;
  for (int k = 0; k < 9; ++k) e[k] = __ddiv_rn(e[k], nrm);
  double A[9], V[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      A[3 * i + j] = dadd(dadd(dmul(e[i], e[j]), dmul(e[3 + i], e[3 + j])), dmul(e[6 + i], e[6 + j]));
  jacobi_eigen<3>(A, V);
  int o[3] = {0, 1, 2};                                 // descending eigenvalue, lowest index on ties
  for (int i = 0; i < 3; ++i)
    for (int j = 2; j > i; --j)
      if (A[4 * o[j]] > A[4 * o[j - 1]]) { const int x = o[j]; o[j] = o[j - 1]; o[j - 1] = x; }
  const double s1 = __dsqrt_rn(fmax(A[4 * o[0]], 0.0)), s2 = __dsqrt_rn(fmax(A[4 * o[1]], 0.0));
  if (!(s2 > dmul(1e-12, s1))) return false;
  double v[3][3];
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) v[i][k] = V[3 * k + o[i]];
  double c[3];
  cross3(v[1], v[2], c);
  if (dot3(v[0], c) < 0.0)
    for (int k = 0; k < 3; ++k) v[2][k] = -v[2][k];
  double u[3][3];
  for (int i = 0; i < 2; ++i)
    for (int k = 0; k < 3; ++k) u[i][k] = dot3(e + 3 * k, v[i]);
  if (!normalise3(u[0])) return false;
  const double pr = dot3(u[0], u[1]);
  for (int k = 0; k < 3; ++k) u[1][k] = dsub(u[1][k], dmul(pr, u[0][k]));
  if (!normalise3(u[1])) return false;
  cross3(u[0], u[1], u[2]);
  // U W = [-u2, u1, u3], U W^T = [u2, -u1, u3]: R = sum_j (U W)_col j v_j^T
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      const double x = dmul(u[0][i], v[1][j]), y = dmul(u[1][i], v[0][j]), z = dmul(u[2][i], v[2][j]);
      Rc[0][3 * i + j] = dadd(dsub(x, y), z);
      Rc[1][3 * i + j] = dadd(dsub(y, x), z);
    }
  for (int k = 0; k < 3; ++k) t[k] = u[2][k];
  return true;
}

// E = [t]x R and the derivatives of E along the 5 refinement directions (thread 0): dE/dw_j = [t]x [e_j]x R,
// dE/dd_j = [b_j]x R with b1 = normalise(t x e_i*) (i* = argmin |t_i|, lowest on ties), b2 = t x b1.
__device__ __noinline__ void linearise(const double* R, const double* t, double* E, double* dE, double* B) {
  double S[9], T[9], M[9];
  skew(t, S);
  mat3(S, R, E);
  for (int j = 0; j < 3; ++j) {
    double ej[3] = {0.0, 0.0, 0.0};
    ej[j] = 1.0;
    skew(ej, T);
    mat3(S, T, M);
    mat3(M, R, dE + 9 * j);
  }
  int im = 0;
  for (int i = 1; i < 3; ++i) if (fabs(t[i]) < fabs(t[im])) im = i;
  double ei[3] = {0.0, 0.0, 0.0};
  ei[im] = 1.0;
  cross3(t, ei, B);
  normalise3(B);
  cross3(t, B, B + 3);
  for (int j = 0; j < 2; ++j) {
    skew(B + 3 * j, T);
    mat3(T, R, dE + 9 * (3 + j));
  }
}

// One LM trial (thread 0): the damped step x, candidate Rn = Exp(x_w) R, tn = normalise(t + x_d1 b1 + x_d2 b2),
// En = [tn]x Rn.  false: no step, or tn is zero.
__device__ __noinline__ bool lm_candidate(const double* J, double lam, const double* R, const double* t,
                                          const double* B, double* Rn, double* tn, double* En) {
  double x[NP];
  if (!lm_solve<NP>(J, lam, x)) return false;
  double X[9];
  rodrigues(x, X);
  mat3(X, R, Rn);
  for (int i = 0; i < 3; ++i) tn[i] = dadd(dadd(t[i], dmul(x[3], B[i])), dmul(x[4], B[3 + i]));
  if (!normalise3(tn)) return false;
  double S[9];
  skew(tn, S);
  mat3(S, Rn, En);
  return true;
}

__global__ void __launch_bounds__(GEO_THREADS) pose_kernel(PoseParams r) {
  __shared__ uint8_t flag[MAX_L];
  __shared__ double red[(GEO_THREADS / 32) * NJ];
  __shared__ double sum[NJ];
  __shared__ double Rc[2][9], tc[3];                   // decomposition
  __shared__ double sR[9], st[3], sE[9], sdE[NP * 9], sB[6];   // current pose and its linearisation
  __shared__ double nR[9], nt[3], nE[9];               // LM candidate
  __shared__ int scan[GEO_THREADS];
  __shared__ int s_total, s_have;
  const int p = blockIdx.x, tid = threadIdx.x;
  int a, b;
  const int n = pair_rows(r, p, a, b);
  const double fx = r.fx, fy = r.fy;

  // ---- decomposition
  if (tid == 0) s_have = decompose(r.E + 9 * (size_t)p, Rc, tc);
  __syncthreads();
  const bool dec = s_have;

  // ---- cheirality of the four candidates (and the usable rows)
  double cg[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  if (dec)
    for (int k = tid; k < n; k += GEO_THREADS) {
      double f1[3], f2[3], X[3];
      if (!rays(r, p, a, b, k, f1, f2)) continue;
      cg[4] = dadd(cg[4], 1.0);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const double tt[3] = {c & 2 ? -tc[0] : tc[0], c & 2 ? -tc[1] : tc[1], c & 2 ? -tc[2] : tc[2]};
        if (triangulate(Rc[c & 1], tt, f1, f2, r.dist, X)) cg[c] = dadd(cg[c], 1.0);
      }
    }
  block_sum<5>(cg, red, sum);
  const int usable = (int)sum[4];
  if (tid == 0) {
    int best = 0;
    for (int c = 1; c < 4; ++c) if (sum[c] > sum[best]) best = c;
    s_have = dec && sum[best] > 0.0;
    if (r.cand_good)
      for (int c = 0; c < 4; ++c) r.cand_good[4 * (size_t)p + c] = (int)sum[c];
    for (int i = 0; i < 9; ++i) sR[i] = Rc[best & 1][i];
    for (int i = 0; i < 3; ++i) st[i] = best & 2 ? -tc[i] : tc[i];
    if (s_have) linearise(sR, st, sE, sdE, sB);
  }
  __syncthreads();
  const bool have = s_have;

  // ---- refinement
  double2 cost = make_double2(0.0, 0.0);                // r^T r before / after
  if (have) {
    const bool refine = r.iters > 0 && usable >= MIN_REFINE_ROWS;
    auto acc_row = [&](int k, double (&acc)[NJ]) {
      double f1[3], f2[3], l[4], s;
      if (!rays(r, p, a, b, k, f1, f2)) return;
      const double res = sampson(sE, f1, f2, fx, fy, l, s);
      double jr[NP];
#pragma unroll
      for (int j = 0; j < NP; ++j) {
        double dl[4];
        const double dnum = epi_terms(sdE + 9 * j, f1, f2, fx, fy, dl);
        jr[j] = s > 0.0 ? __ddiv_rn(dsub(dnum, __ddiv_rn(dmul(res, dot4(l, dl)), s)), s) : 0.0;
      }
      lm_add<NP>(acc, jr, res);
    };
    auto cost_row = [&](int k, double& c) {
      double f1[3], f2[3], l[4], s;
      if (!rays(r, p, a, b, k, f1, f2)) return;
      const double res = sampson(nE, f1, f2, fx, fy, l, s);
      c = dadd(c, dmul(res, res));
    };
    auto step = [&](const double* J, double lam) { return lm_candidate(J, lam, sR, st, sB, nR, nt, nE); };
    auto commit = [&] {
      for (int i = 0; i < 9; ++i) sR[i] = nR[i];
      for (int i = 0; i < 3; ++i) st[i] = nt[i];
      linearise(sR, st, sE, sdE, sB);
    };
    cost = lm_refine<NP>(n, refine, r.iters, red, sum, acc_row, cost_row, step, commit);
  }

  // ---- final pass: cheirality of the refined pose, mask, points, compaction
  for (int k = tid; k < r.L; k += GEO_THREADS) {
    double f1[3], f2[3], X[3] = {0.0, 0.0, 0.0};
    bool good = false;
    if (have && k < n && rays(r, p, a, b, k, f1, f2)) good = triangulate(sR, st, f1, f2, r.dist, X);
    if (k < n) flag[k] = good;
    if (r.mask) r.mask[(size_t)p * r.L + k] = good;
    if (r.points) {
      float* o = r.points + ((size_t)p * r.L + k) * 3;
      o[0] = good ? __double2float_rn(X[0]) : 0.f;
      o[1] = good ? __double2float_rn(X[1]) : 0.f;
      o[2] = good ? __double2float_rn(X[2]) : 0.f;
    }
  }
  if (tid < 9) r.R[9 * (size_t)p + tid] = have ? sR[tid] : 0.0;
  if (tid < 3) r.t[3 * (size_t)p + tid] = have ? st[tid] : 0.0;
  if (r.rms && tid < 2) {
    const double c = tid == 0 ? cost.x : cost.y;
    r.rms[2 * (size_t)p + tid] = have && usable > 0 ? __dsqrt_rn(__ddiv_rn(c, (double)usable)) : 0.0;
  }
  __syncthreads();
  const int total = compact_rows(flag, n, r.L, p, r.pairs, r.pair_scores, r.out_pairs, r.out_scores, scan, &s_total);
  if (tid == 0) r.out_counts[p] = total;
}

}  // namespace
}  // namespace sslam

using namespace sslam;

extern "C" int sslam_recover_pose(const float* kpts1, int F1, const float* kpts2, int F2, const int32_t* pair_index,
                                  int P, int N, int M, const double* E, const int32_t* pairs,
                                  const float* pair_scores, const int32_t* counts, int L, double fx, double fy,
                                  double cx, double cy, double distance_thresh, int refine_iters, double* R,
                                  double* t, int32_t* cand_good, double* rms, float* points, int32_t* out_pairs,
                                  float* out_scores, int32_t* out_counts, uint8_t* pose_mask, void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  const double K[4] = {fx, fy, cx, cy};
  rc = check_list_args("recover_pose", P, N, M, L, F1, F2, pair_index,
                       kpts1 && kpts2 && E && pairs && pair_scores && counts && R && t && out_pairs && out_scores &&
                           out_counts,
                       nullptr, &refine_iters, "distance_thresh", distance_thresh, K);
  if (rc || P == 0) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  PoseParams r{kpts1, kpts2, F1, F2, pair_index, P, N, M, E, pairs, pair_scores, counts, L,
               fx, fy, cx, cy, distance_thresh, refine_iters, R, t, cand_good, rms, points,
               out_pairs, out_scores, out_counts, pose_mask};
  SSLAM_LAUNCH(KK_POSE, stream, pose_kernel<<<P, GEO_THREADS, 0, stream>>>(r));
  return SSLAM_OK;
}
