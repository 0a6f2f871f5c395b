// Helpers shared by the per-pair geometry kernels (ransac.cu, pose.cu, pnp.cu, triangulate.cu): the
// argument checks of the list entries, the padded match-list accessors, the splitmix64 row sampler,
// correctly rounded double arithmetic, 3x3 helpers and Rodrigues, calibrated rays and midpoint
// triangulation, the fixed-order block reductions, cyclic Jacobi, the Levenberg-Marquardt loop, the
// order-preserving compaction into the matcher's list format and the RANSAC workspace layout.
#pragma once

#include "common.cuh"

namespace sslam {
namespace {

constexpr int GEO_THREADS = 256;      // threads of the one-CTA-per-pair kernels (refit, pose)
constexpr int MAX_L = 16384;          // list stride limit (row flags live in shared memory)
constexpr int MAX_ITERS = 65536;      // RANSAC samples per list
constexpr int MAX_REFINE = 100;       // Levenberg-Marquardt trials
constexpr int MAX_DRAWS = 32;         // sampler draws per sample (redraws included)
// Levenberg-Marquardt damping schedule: lambda starts at LM_LAMBDA0 times the mean of diag(J^T J); an
// accepted trial divides it by LM_LAMBDA_STEP, a rejected one multiplies it by LM_LAMBDA_STEP.
constexpr double LM_LAMBDA0 = 1e-3;
constexpr double LM_LAMBDA_STEP = 10.0;

// Checks shared by the match-list entries; SSLAM_OK or the code to return, the message prefixed by fn.
// iters, refine_iters and the intrinsics K = {fx, fy, cx, cy} are checked where the entry takes them (not
// null); thresh (named thresh_name) must be finite and > 0.  With P == 0 nothing else is needed, so
// pointers (every required pointer set) and the banks are checked only for P > 0.
inline int check_list_args(const char* fn, int P, int N, int M, int L, int F1, int F2, const void* pair_index,
                           bool pointers, const int* iters, const int* refine_iters, const char* thresh_name,
                           double thresh, const double* K) {
  SSLAM_REQUIRE(P >= 0 && N >= 0 && M >= 0 && L >= 0, SSLAM_EINVAL, "%s: bad size", fn);
  SSLAM_REQUIRE(L <= MAX_L, SSLAM_EINVAL, "%s: list stride %d > %d", fn, L, MAX_L);
  SSLAM_REQUIRE(!iters || (*iters >= 1 && *iters <= MAX_ITERS), SSLAM_EINVAL, "%s: iters=%d (need 1..%d)", fn,
                *iters, MAX_ITERS);
  SSLAM_REQUIRE(!refine_iters || (*refine_iters >= 0 && *refine_iters <= MAX_REFINE), SSLAM_EINVAL,
                "%s: refine_iters=%d (need 0..%d)", fn, *refine_iters, MAX_REFINE);
  SSLAM_REQUIRE(thresh > 0.0 && isfinite(thresh), SSLAM_EINVAL, "%s: %s must be finite and > 0", fn, thresh_name);
  SSLAM_REQUIRE(!K || (K[0] > 0.0 && K[1] > 0.0 && isfinite(K[0]) && isfinite(K[1]) && isfinite(K[2]) &&
                       isfinite(K[3])), SSLAM_EINVAL, "%s: need fx, fy > 0 and finite intrinsics", fn);
  if (P == 0) return SSLAM_OK;
  SSLAM_REQUIRE(pointers, SSLAM_EINVAL, "%s: null pointer", fn);
  SSLAM_REQUIRE(F1 > 0 && F2 > 0 && (pair_index || (F1 >= P && F2 >= P)), SSLAM_EINVAL,
                "%s: banks hold %d / %d sets but %d implicit lists were requested", fn, F1, F2, P);
  return SSLAM_OK;
}

// Rows of pair p, clamped to the list stride; 0 when the pair's frame ids are out of range.  Pm has the
// fields k1, k2, F1, F2, pair_index, N, M, pairs, counts, L of the C ABI's list arguments.
template <class Pm>
__device__ __forceinline__ int pair_rows(const Pm& r, int p, int& a, int& b) {
  a = p; b = p;
  if (r.pair_index) { a = r.pair_index[2 * p]; b = r.pair_index[2 * p + 1]; }
  if (a < 0 || a >= r.F1 || b < 0 || b >= r.F2) return 0;
  return min(max(r.counts[p], 0), r.L);
}

// Correspondence of row k as (x1, y1, x2, y2); NaN (never an inlier, degenerate sample) when the
// row's keypoint indices are out of range.
template <class Pm>
__device__ __forceinline__ float4 corr(const Pm& r, int p, int a, int b, int k) {
  const int2 ij = reinterpret_cast<const int2*>(r.pairs)[(size_t)p * r.L + k];
  if (ij.x < 0 || ij.x >= r.N || ij.y < 0 || ij.y >= r.M) {
    const float nan = __int_as_float(0x7fc00000);
    return make_float4(nan, nan, nan, nan);
  }
  const float2 u = reinterpret_cast<const float2*>(r.k1)[(size_t)a * r.N + ij.x];
  const float2 v = reinterpret_cast<const float2*>(r.k2)[(size_t)b * r.M + ij.y];
  return make_float4(u.x, u.y, v.x, v.y);
}

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dadd_rn(a, -b); }

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

__device__ __forceinline__ double dot3(const double* a, const double* b) {
  return dadd(dadd(dmul(a[0], b[0]), dmul(a[1], b[1])), dmul(a[2], b[2]));
}

// C = A B (3x3, row-major).
__device__ __forceinline__ void mat3(const double* A, const double* B, double* C) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      C[3 * i + j] = dadd(dadd(dmul(A[3 * i], B[j]), dmul(A[3 * i + 1], B[3 + j])), dmul(A[3 * i + 2], B[6 + j]));
}

__device__ __forceinline__ void skew(const double* v, double* S) {
  S[0] = 0.0; S[1] = -v[2]; S[2] = v[1];
  S[3] = v[2]; S[4] = 0.0; S[5] = -v[0];
  S[6] = -v[1]; S[7] = v[0]; S[8] = 0.0;
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
  c[0] = dsub(dmul(a[1], b[2]), dmul(a[2], b[1]));
  c[1] = dsub(dmul(a[2], b[0]), dmul(a[0], b[2]));
  c[2] = dsub(dmul(a[0], b[1]), dmul(a[1], b[0]));
}

// Exp(w) by Rodrigues: I + sin(th) K + (1 - cos(th)) K^2, K = [w / th]x, th = |w|; I when th = 0.
__device__ __forceinline__ void rodrigues(const double* w, double* X) {
  for (int i = 0; i < 9; ++i) X[i] = (i % 4 == 0) ? 1.0 : 0.0;
  const double th = __dsqrt_rn(dot3(w, w));
  if (th > 0.0) {
    const double k[3] = {__ddiv_rn(w[0], th), __ddiv_rn(w[1], th), __ddiv_rn(w[2], th)};
    double K[9], K2[9];
    skew(k, K);
    mat3(K, K, K2);
    const double sn = sin(th), cs = dsub(1.0, cos(th));
    for (int i = 0; i < 9; ++i) X[i] = dadd(dadd(X[i], dmul(sn, K[i])), dmul(cs, K2[i]));
  }
}

// Normalised rays (K^-1 x) of row k; false when the row is not usable (a keypoint index out of range, or
// a coordinate that is not finite).  Pm: the list fields of pair_rows / corr and fx, fy, cx, cy.
template <class Pm>
__device__ __forceinline__ bool rays(const Pm& r, int p, int a, int b, int k, double f1[3], double f2[3]) {
  const float4 q = corr(r, p, a, b, k);
  if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z) && isfinite(q.w))) return false;
  f1[0] = __ddiv_rn(dsub(q.x, r.cx), r.fx); f1[1] = __ddiv_rn(dsub(q.y, r.cy), r.fy); f1[2] = 1.0;
  f2[0] = __ddiv_rn(dsub(q.z, r.cx), r.fx); f2[1] = __ddiv_rn(dsub(q.w, r.cy), r.fy); f2[2] = 1.0;
  return true;
}

// Midpoint of the rays f1, f2 under (R, t), x2 ~ R x1 + t: the depths z1, z2 minimising |z1 u + t - z2 f2|
// with u = R f1, X = z1 f1 (camera-1 frame).  Returns whether the rays are not parallel, den > 1e-12 a c.
__device__ __forceinline__ bool midpoint(const double* R, const double* t, const double f1[3], const double f2[3],
                                         double X[3]) {
  const double u[3] = {dot3(R, f1), dot3(R + 3, f1), dot3(R + 6, f1)};
  const double a = dot3(u, u), b = dot3(u, f2), c = dot3(f2, f2), d = dot3(u, t), e = dot3(f2, t);
  const double den = dsub(dmul(a, c), dmul(b, b));
  const double z1 = __ddiv_rn(dsub(dmul(b, e), dmul(c, d)), den);
  X[0] = dmul(z1, f1[0]); X[1] = dmul(z1, f1[1]); X[2] = z1;
  return den > dmul(dmul(1e-12, a), c);
}

// Triangulation of one row under (R, t) with cv2.recoverPose's cheirality: good iff the rays are not
// parallel, 0 < z1 < dist and 0 < (R X + t)_z < dist.
__device__ __forceinline__ bool triangulate(const double* R, const double* t, const double f1[3],
                                            const double f2[3], double dist, double X[3]) {
  const bool apart = midpoint(R, t, f1, f2, X);
  const double z1 = X[2];
  const double z2 = dadd(dot3(R + 6, X), t[2]);
  return apart && z1 > 0.0 && z1 < dist && z2 > 0.0 && z2 < dist;
}

// Fixed-order block sum of R doubles per thread over GEO_THREADS threads: warp butterflies, then warps
// in order.
template <int R>
__device__ __forceinline__ void block_sum(double (&v)[R], double* red /* [GEO_THREADS/32][R] */,
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
    for (int w = 1; w < GEO_THREADS / 32; ++w) s = dadd(s, red[w * R + threadIdx.x]);
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------- Levenberg-Marquardt
// Accumulators of an NP-parameter refinement: J^T J upper triangle, J^T r, r^T r.
constexpr int lm_nj(int np) { return np * (np + 1) / 2 + np + 1; }

// The starting damping of the accumulators Js: LM_LAMBDA0 times the mean of diag(J^T J).
template <int NP>
__device__ __forceinline__ double lm_lambda0(const double* Js) {
  double d = 0.0;
  int q = 0;
  for (int i = 0; i < NP; q += NP - i, ++i) d = dadd(d, Js[q]);
  return dmul(LM_LAMBDA0, __ddiv_rn(d, (double)NP));
}

// Adds one residual r with Jacobian row j to the accumulators.
template <int NP>
__device__ __forceinline__ void lm_add(double (&acc)[lm_nj(NP)], const double* j, double r) {
  int q = 0;
#pragma unroll
  for (int i = 0; i < NP; ++i)
#pragma unroll
    for (int k = i; k < NP; ++k, ++q) acc[q] = dadd(acc[q], dmul(j[i], j[k]));
#pragma unroll
  for (int i = 0; i < NP; ++i) acc[q + i] = dadd(acc[q + i], dmul(j[i], r));
  acc[lm_nj(NP) - 1] = dadd(acc[lm_nj(NP) - 1], dmul(r, r));
}

// The damped step (thread 0): (J^T J + lam diag(J^T J)) x = -J^T r by Cholesky.  false: the system is not
// positive definite or the step is not finite.
template <int NP>
__device__ __forceinline__ bool lm_solve(const double* Js, double lam, double x[NP]) {
  double A[NP][NP], Lc[NP][NP];
  int q = 0;
  for (int i = 0; i < NP; ++i)
    for (int j = i; j < NP; ++j, ++q) A[i][j] = A[j][i] = Js[q];
  for (int i = 0; i < NP; ++i) A[i][i] = dadd(A[i][i], dmul(lam, A[i][i]));
  for (int j = 0; j < NP; ++j) {
    double d = A[j][j];
    for (int k = 0; k < j; ++k) d = dsub(d, dmul(Lc[j][k], Lc[j][k]));
    if (!(d > 0.0)) return false;
    Lc[j][j] = __dsqrt_rn(d);
    for (int i = j + 1; i < NP; ++i) {
      double s = A[i][j];
      for (int k = 0; k < j; ++k) s = dsub(s, dmul(Lc[i][k], Lc[j][k]));
      Lc[i][j] = __ddiv_rn(s, Lc[j][j]);
    }
  }
  for (int i = 0; i < NP; ++i) {                        // L y = -J^T r
    double s = -Js[NP * (NP + 1) / 2 + i];
    for (int k = 0; k < i; ++k) s = dsub(s, dmul(Lc[i][k], x[k]));
    x[i] = __ddiv_rn(s, Lc[i][i]);
  }
  for (int i = NP - 1; i >= 0; --i) {                   // L^T x = y
    double s = x[i];
    for (int k = i + 1; k < NP; ++k) s = dsub(s, dmul(Lc[k][i], x[k]));
    x[i] = __ddiv_rn(s, Lc[i][i]);
  }
  bool ok = true;
  for (int i = 0; i < NP; ++i) ok &= isfinite(x[i]);
  return ok;
}

// Levenberg-Marquardt over the rows k < n, every thread of the block (GEO_THREADS) calls it.  Linearise
// (acc_row(k, acc) adds row k's terms with lm_add, or skips the row), lam = lm_lambda0; then, when
// `refine`, `iters` trials: step(Jsum, lam) forms the candidate on thread 0 (false: no step), cost_row(k, c)
// adds row k's squared residual under it, a strictly lower cost is accepted (commit() on thread 0,
// lam / LM_LAMBDA_STEP, relinearise before the next trial), anything else sets lam * LM_LAMBDA_STEP.  All
// sums are fixed-order block sums (red, sum: block_sum scratch of lm_nj(NP) doubles per warp and in all).
// Returns (cost0, cost): r^T r at the start and at the end.
template <int NP, class AccRow, class CostRow, class Step, class Commit>
__device__ __forceinline__ double2 lm_refine(int n, bool refine, int iters, double* red, double* sum,
                                             AccRow acc_row, CostRow cost_row, Step step, Commit commit) {
  constexpr int NJ = lm_nj(NP);
  __shared__ double Jsum[NJ];
  __shared__ double s_cost, s_lam;
  const int tid = threadIdx.x;
  double cost0 = 0.0;
  bool relin = true;
  for (int it = -1; it < (refine ? iters : 0); ++it) {
    if (relin) {                                        // J^T J, J^T r, r^T r at the current state
      double acc[NJ];
#pragma unroll
      for (int i = 0; i < NJ; ++i) acc[i] = 0.0;
      for (int k = tid; k < n; k += GEO_THREADS) acc_row(k, acc);
      block_sum<NJ>(acc, red, sum);
      if (tid == 0) {
        for (int i = 0; i < NJ; ++i) Jsum[i] = sum[i];
        if (it < 0) {
          s_cost = sum[NJ - 1];
          s_lam = lm_lambda0<NP>(sum);
        }
      }
      __syncthreads();
      if (it < 0) cost0 = s_cost;
      relin = false;
      if (it < 0) continue;
    }
    bool stepped = false;
    if (tid == 0) stepped = step(Jsum, s_lam);
    bool accept = false;
    if (__syncthreads_or(stepped)) {
      double c1[1] = {0.0};
      for (int k = tid; k < n; k += GEO_THREADS) cost_row(k, c1[0]);
      block_sum<1>(c1, red, sum);
      accept = sum[0] < s_cost;
    }
    __syncthreads();
    if (tid == 0) {
      if (accept) {
        s_cost = sum[0];
        s_lam = __ddiv_rn(s_lam, LM_LAMBDA_STEP);
        commit();
      } else {
        s_lam = dmul(s_lam, LM_LAMBDA_STEP);
      }
    }
    __syncthreads();
    relin = accept && it + 1 < iters;
  }
  return make_double2(cost0, s_cost);
}

// Cyclic Jacobi on a symmetric NxN (one thread, shared or local memory): on return the diagonal of A
// holds the eigenvalues and column i of V the eigenvector of A[i][i].
template <int N>
__device__ __forceinline__ void jacobi_eigen(double* A, double* V) {
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
}

// The eigenvector of the smallest eigenvalue of a symmetric NxN (lowest index on ties) in v_out.
template <int N>
__device__ void jacobi_smallest(double* A, double* V, double* v_out) {
  jacobi_eigen<N>(A, V);
  int m = 0;
  for (int i = 1; i < N; ++i) if (A[(N + 1) * i] < A[(N + 1) * m]) m = i;
  for (int k = 0; k < N; ++k) v_out[k] = V[N * k + m];
}

// Order-preserving compaction of the rows k < n with flag[k] set into list p of the matcher's format
// (rows (i, j) -1 padded, scores 0 padded, stride L); every thread of the block calls it.  scan: int
// [GEO_THREADS] shared scratch, s_total: shared.  Returns the number of rows kept.
__device__ __forceinline__ int compact_rows(const uint8_t* flag, int n, int L, int p, const int32_t* pairs,
                                            const float* pair_scores, int32_t* out_pairs, float* out_scores,
                                            int* scan, int* s_total) {
  const int tid = threadIdx.x;
  const int seg = (n + GEO_THREADS - 1) / GEO_THREADS;
  const int beg = min(n, tid * seg), end = min(n, beg + seg);
  int cnt = 0;
  for (int k = beg; k < end; ++k) cnt += flag[k];
  scan[tid] = cnt;
  __syncthreads();
  for (int o = 1; o < GEO_THREADS; o <<= 1) {
    const int v = (tid >= o) ? scan[tid - o] : 0;
    __syncthreads();
    scan[tid] += v;
    __syncthreads();
  }
  int pos = scan[tid] - cnt;
  if (tid == GEO_THREADS - 1) *s_total = scan[GEO_THREADS - 1];
  __syncthreads();
  const int total = *s_total;
  const int2* in_pr = reinterpret_cast<const int2*>(pairs) + (size_t)p * L;
  const float* in_sc = pair_scores + (size_t)p * L;
  int2* pr = reinterpret_cast<int2*>(out_pairs) + (size_t)p * L;
  float* ps = out_scores + (size_t)p * L;
  for (int k = beg; k < end; ++k)
    if (flag[k]) { pr[pos] = in_pr[k]; ps[pos] = in_sc[k]; ++pos; }
  for (int k = total + tid; k < L; k += GEO_THREADS) { pr[k] = make_int2(-1, -1); ps[k] = 0.f; }
  return total;
}

// Workspace of the three-launch RANSAC kernels (ransac.cu, pnp.cu): per-slot inlier counts int32
// [P, slots], the best slot [P], the best slot's pre-refit mask [P, L], the fp32 hypotheses
// [P, slots, floats]; each part starts at a 256-byte boundary.
struct WsLayout { size_t count, best, mask, hyp, total; };

inline WsLayout ws_layout(int P, int L, int iters, int slots_per_sample, int floats) {
  const size_t slots = (size_t)iters * slots_per_sample;
  WsLayout w;
  w.count = 0;
  w.best = align_up((size_t)P * slots * 4, 256);
  w.mask = w.best + align_up((size_t)P * 4, 256);
  w.hyp = w.mask + align_up((size_t)P * L, 256);
  w.total = w.hyp + align_up((size_t)P * slots * floats * 4, 256);
  return w;
}

}  // namespace
}  // namespace sslam
