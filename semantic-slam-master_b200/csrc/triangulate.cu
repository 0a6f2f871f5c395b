// Triangulation of match lists under a known relative pose: one CTA (256 threads) per list, one launch, no
// workspace, no atomics.  Each row is worked on one thread, in double with correctly rounded operations:
//
//   midpoint     the rays f1 = K^-1 x1, f2 = K^-1 x2 and their midpoint X in the camera-a frame (pose.cu's
//                cheirality triangulation, with its "rays not parallel" test den > 1e-12 a c)
//   refinement   up to refine_iters Levenberg-Marquardt trials on X (3 DOF) over the 4 pixel residuals
//                pi(X) - x1, pi(R X + t) - x2, in the thread's registers, with the damping schedule of
//                lm_refine; a candidate with a depth <= 0 in either camera is rejected
//   gates        kept iff the rays are not parallel, 0 < z_a, z_b < dist, the parallax cosine between X and
//                X - C_b (C_b = -R^T t) is <= max_cos, and the squared reprojection error is < t^2 in both
//                views
//
// The kept rows are compacted into the matcher's list format.  Every result is a function of the list's own
// inputs, never of its position in the batch.  oracle/triangulate.py restates every step in the same order.
#include "geometry.cuh"

namespace sslam {
namespace {

constexpr int NP = 3;                 // refinement parameters: X
constexpr int NJ = lm_nj(NP);

struct TriParams {
  const float* k1; const float* k2;          // [F1,N,2], [F2,M,2]
  int F1, F2;
  const int32_t* pair_index;                 // [P,2] or null
  int P, N, M;
  const int32_t* pairs; const float* pair_scores; const int32_t* counts;   // [P,L,2], [P,L], [P]
  int L;
  const double* R; const double* t;          // [P,9], [P,3]
  double fx, fy, cx, cy, t2, max_cos, dist;
  int iters;
  float* points;                             // [P,L,3] or null
  int32_t* out_pairs; float* out_scores; int32_t* out_counts; uint8_t* mask;
};

// Pixel residuals of X (camera a) against q = (x1, y1, x2, y2) in both views, res = (u_a, v_a, u_b, v_b),
// the depths z_a, z_b, and optionally the Jacobian rows d res / d X.
__device__ __forceinline__ void tri_residuals(const double* R, const double* t, const double X[3], const float4& q,
                                              double fx, double fy, double cx, double cy, double res[4],
                                              double z[2], double (*J)[NP]) {
  const double Y[3] = {dadd(dot3(R, X), t[0]), dadd(dot3(R + 3, X), t[1]), dadd(dot3(R + 6, X), t[2])};
  const double* V[2] = {X, Y};
  const double uv[2][2] = {{q.x, q.y}, {q.z, q.w}};
#pragma unroll
  for (int v = 0; v < 2; ++v) {
    const double iz = __ddiv_rn(1.0, V[v][2]);
    const double pu = dmul(V[v][0], iz), pv = dmul(V[v][1], iz);
    z[v] = V[v][2];
    res[2 * v] = dsub(dadd(dmul(fx, pu), cx), uv[v][0]);
    res[2 * v + 1] = dsub(dadd(dmul(fy, pv), cy), uv[v][1]);
    if (!J) continue;
    const double gu[3] = {dmul(fx, iz), 0.0, -dmul(dmul(fx, pu), iz)};
    const double gv[3] = {0.0, dmul(fy, iz), -dmul(dmul(fy, pv), iz)};
    for (int k = 0; k < 3; ++k) {
      if (v == 0) {
        J[0][k] = gu[k];
        J[1][k] = gv[k];
      } else {                                         // d Y / d X = R
        const double col[3] = {R[k], R[3 + k], R[6 + k]};
        J[2][k] = dot3(gu, col);
        J[3][k] = dot3(gv, col);
      }
    }
  }
}

// J^T J, J^T r, r^T r of the 4 residuals at X.
__device__ __forceinline__ void tri_linearise(const double* R, const double* t, const double X[3], const float4& q,
                                              double fx, double fy, double cx, double cy, double (&acc)[NJ]) {
  double res[4], z[2], J[4][NP];
  tri_residuals(R, t, X, q, fx, fy, cx, cy, res, z, J);
#pragma unroll
  for (int i = 0; i < NJ; ++i) acc[i] = 0.0;
#pragma unroll
  for (int e = 0; e < 4; ++e) lm_add<NP>(acc, J[e], res[e]);
}

// Whether one usable row (rays f1, f2, pixels q) is kept; X: its final point.
__device__ __forceinline__ bool tri_row(const TriParams& r, const double* R, const double* t, const double f1[3],
                                        const double f2[3], const float4 q, double X[3]) {
  const double fx = r.fx, fy = r.fy, cx = r.cx, cy = r.cy;
  const bool apart = midpoint(R, t, f1, f2, X);
  if (!apart) return false;
  if (r.iters > 0) {
    double acc[NJ];
    tri_linearise(R, t, X, q, fx, fy, cx, cy, acc);
    double cost = acc[NJ - 1];
    double lam = lm_lambda0<NP>(acc);
    for (int it = 0; it < r.iters; ++it) {
      double x[NP];
      bool accept = false;
      double Xn[3], c = 0.0;
      if (lm_solve<NP>(acc, lam, x)) {
        for (int i = 0; i < 3; ++i) Xn[i] = dadd(X[i], x[i]);
        double res[4], z[2];
        tri_residuals(R, t, Xn, q, fx, fy, cx, cy, res, z, nullptr);
        for (int e = 0; e < 4; ++e) c = dadd(c, dmul(res[e], res[e]));
        accept = z[0] > 0.0 && z[1] > 0.0 && c < cost;
      }
      if (accept) {
        for (int i = 0; i < 3; ++i) X[i] = Xn[i];
        cost = c;
        lam = __ddiv_rn(lam, LM_LAMBDA_STEP);
        if (it + 1 < r.iters) tri_linearise(R, t, X, q, fx, fy, cx, cy, acc);
      } else {
        lam = dmul(lam, LM_LAMBDA_STEP);
      }
    }
  }
  double res[4], z[2];
  tri_residuals(R, t, X, q, fx, fy, cx, cy, res, z, nullptr);
  const double cb[3] = {-dadd(dadd(dmul(R[0], t[0]), dmul(R[3], t[1])), dmul(R[6], t[2])),
                        -dadd(dadd(dmul(R[1], t[0]), dmul(R[4], t[1])), dmul(R[7], t[2])),
                        -dadd(dadd(dmul(R[2], t[0]), dmul(R[5], t[1])), dmul(R[8], t[2]))};
  const double v[3] = {dsub(X[0], cb[0]), dsub(X[1], cb[1]), dsub(X[2], cb[2])};
  const double cosp = __ddiv_rn(dot3(X, v), dmul(__dsqrt_rn(dot3(X, X)), __dsqrt_rn(dot3(v, v))));
  const double ea = dadd(dmul(res[0], res[0]), dmul(res[1], res[1]));
  const double eb = dadd(dmul(res[2], res[2]), dmul(res[3], res[3]));
  return z[0] > 0.0 && z[0] < r.dist && z[1] > 0.0 && z[1] < r.dist && cosp <= r.max_cos && ea < r.t2 &&
         eb < r.t2;
}

__global__ void __launch_bounds__(GEO_THREADS) triangulate_kernel(TriParams r) {
  __shared__ uint8_t flag[MAX_L];
  __shared__ double sRt[12];                           // R row-major, t
  __shared__ int scan[GEO_THREADS];
  __shared__ int s_total, s_have;
  const int p = blockIdx.x, tid = threadIdx.x;
  int a, b;
  const int n = pair_rows(r, p, a, b);
  if (tid < 12) sRt[tid] = tid < 9 ? r.R[9 * (size_t)p + tid] : r.t[3 * (size_t)p + tid - 9];
  __syncthreads();
  if (tid == 0) {                                      // a non-finite entry, or R all zero: no pose
    bool fin = true, nonzero = false;
    for (int i = 0; i < 12; ++i) fin &= isfinite(sRt[i]);
    for (int i = 0; i < 9; ++i) nonzero |= sRt[i] != 0.0;
    s_have = fin && nonzero;
  }
  __syncthreads();
  const bool have = s_have;
  for (int k = tid; k < r.L; k += GEO_THREADS) {
    double f1[3], f2[3], X[3] = {0.0, 0.0, 0.0};
    bool good = false;
    if (have && k < n && rays(r, p, a, b, k, f1, f2))
      good = tri_row(r, sRt, sRt + 9, f1, f2, corr(r, p, a, b, k), X);
    if (k < n) flag[k] = good;
    if (r.mask) r.mask[(size_t)p * r.L + k] = good;
    if (r.points) {
      float* o = r.points + ((size_t)p * r.L + k) * 3;
      o[0] = good ? __double2float_rn(X[0]) : 0.f;
      o[1] = good ? __double2float_rn(X[1]) : 0.f;
      o[2] = good ? __double2float_rn(X[2]) : 0.f;
    }
  }
  __syncthreads();
  const int total = compact_rows(flag, n, r.L, p, r.pairs, r.pair_scores, r.out_pairs, r.out_scores, scan, &s_total);
  if (tid == 0) r.out_counts[p] = total;
}

}  // namespace
}  // namespace sslam

using namespace sslam;

extern "C" int sslam_triangulate(const float* kpts1, int F1, const float* kpts2, int F2, const int32_t* pair_index,
                                 int P, int N, int M, const int32_t* pairs, const float* pair_scores,
                                 const int32_t* counts, int L, const double* R, const double* t, double fx, double fy,
                                 double cx, double cy, double threshold, double max_parallax_cos,
                                 double distance_thresh, int refine_iters, float* points, int32_t* out_pairs,
                                 float* out_scores, int32_t* out_counts, uint8_t* mask, void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  SSLAM_REQUIRE(max_parallax_cos >= 0.0 && max_parallax_cos <= 1.0, SSLAM_EINVAL,
                "triangulate: max_parallax_cos must lie in [0, 1]");
  SSLAM_REQUIRE(distance_thresh > 0.0, SSLAM_EINVAL, "triangulate: distance_thresh must be > 0");
  const double K[4] = {fx, fy, cx, cy};
  rc = check_list_args("triangulate", P, N, M, L, F1, F2, pair_index,
                       kpts1 && kpts2 && pairs && pair_scores && counts && R && t && out_pairs && out_scores &&
                           out_counts,
                       nullptr, &refine_iters, "threshold", threshold, K);
  if (rc || P == 0) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  TriParams r{kpts1, kpts2, F1, F2, pair_index, P, N, M, pairs, pair_scores, counts, L, R, t,
              fx, fy, cx, cy, threshold * threshold, max_parallax_cos, distance_thresh, refine_iters, points,
              out_pairs, out_scores, out_counts, mask};
  SSLAM_LAUNCH(KK_TRIANGULATE, stream, triangulate_kernel<<<P, GEO_THREADS, 0, stream>>>(r));
  return SSLAM_OK;
}
