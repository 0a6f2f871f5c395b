// Sliding-window bundle adjustment: one CTA (256 threads) per window of W <= 8 posed frames, one launch, no
// atomics.  The poses of the free frames (the last W - fixed) and the points of the window's tracks are refined
// jointly on the pixel error of every used observation, in double with correctly rounded operations (Rodrigues'
// sin / cos aside):
//
//   used set     fixed at the start: observation (n, w) is used when its slot and keypoint index are in range,
//                the keypoint and the point are finite and the depth is > 0; track n is used when n < counts
//                and it has >= 2 such observations (observations of other tracks are not used either)
//   cost         sum of rho(|r|^2) over the used observations, r = pi(R_w X_n + t_w) - x, Huber rho with IRLS
//                weight min(1, delta / |r|) at the linearisation point (delta = inf: plain least squares)
//   step         R_w <- Exp(w_w) R_w, t_w <- t_w + d_w (free frames), X_n <- X_n + dX_n; Levenberg-Marquardt with
//                lm_refine's schedule and Marquardt damping H_ii (1 + lambda) on pose and point blocks; each
//                trial reduces to the free poses by the Schur complement S = U - sum_n W_n V_n^-1 W_n^T, solves
//                S by a dense Cholesky and back-substitutes per track; a candidate with a used observation at
//                depth <= 0 is rejected, a strictly lower cost accepted
//
// Tracks are visited in chunks of BA_CHUNK, one lane per (track, frame): the 8 lanes of a track sum their
// terms in ascending frame order by shuffles, stage the pose-side terms in shared memory, and each thread then
// owns fixed entries of U / S and sums the chunk's tracks in ascending order, so every sum has one order and
// a window's result does not depend on its position in the batch.  The points live in a workspace (double,
// current and candidate) with the used-observation bits.  oracle/bundle_adjust.py restates every step.
#include "geometry.cuh"

namespace sslam {
namespace {

constexpr int MAX_WINDOW = 8;
constexpr int MAX_TRACKS = 65536;
constexpr int BA_CHUNK = GEO_THREADS / MAX_WINDOW;   // 32 tracks per chunk
constexpr int MAX_NP = 6 * (MAX_WINDOW - 1);         // free pose parameters (at least one frame is held)
constexpr int SLOT = 27;                             // staged doubles per (track, frame): U (21) + b_pose (6), or Z (18) + g (3)
constexpr int MAX_OWN = (MAX_NP * (MAX_NP + 1) / 2 + MAX_NP + GEO_THREADS - 1) / GEO_THREADS;
constexpr size_t STAGE_BYTES = sizeof(double) * BA_CHUNK * MAX_WINDOW * SLOT;   // 55 296 B, also holds S
static_assert(MAX_NP * MAX_NP <= BA_CHUNK * MAX_WINDOW * SLOT, "S must fit in the staging buffer");

struct BaParams {
  const float* kpts; int F, K;                  // [F,K,2]
  const int32_t* frame_index;                   // [P,W]
  int P, W, N;
  const int32_t* obs; const float* points; const int32_t* counts;   // [P,N,W], [P,N,3], [P]
  const double* R; const double* t;             // [P,W,9], [P,W,3]
  double fx, fy, cx, cy, huber, t2;
  int fixed, iters;
  double* R_out; double* t_out; float* points_out; double* rms; int32_t* accepted; uint8_t* mask;
  uint8_t* ws; size_t ws_window;
};

// Workspace of one window: points in double, [2][N][3] (current / candidate), then one byte of used-observation
// bits per track.
inline size_t ws_window_bytes(int N) { return align_up((size_t)N * (2 * 3 * sizeof(double) + 1), 256); }

// Residual of X under P = (R row-major, t) against (u, v), the depth, and optionally the Jacobians along the
// pose (w, d) (R <- Exp(w) R, t <- t + d: dY/dw_j = e_j x (R X), dY/dd = I) and along X (dY/dX = R).
__device__ __forceinline__ void ba_project(const double* P, const double X[3], double u, double v, double fx,
                                           double fy, double cx, double cy, double res[2], double& z,
                                           double (*Jp)[6], double (*Jx)[3]) {
  const double rx[3] = {dot3(P, X), dot3(P + 3, X), dot3(P + 6, X)};
  const double xc = dadd(rx[0], P[9]), yc = dadd(rx[1], P[10]), zc = dadd(rx[2], P[11]);
  z = zc;
  const double iz = __ddiv_rn(1.0, zc);
  const double pu = dmul(xc, iz), pv = dmul(yc, iz);
  res[0] = dsub(dadd(dmul(fx, pu), cx), u);
  res[1] = dsub(dadd(dmul(fy, pv), cy), v);
  if (!Jx) return;
  const double gu[3] = {dmul(fx, iz), 0.0, -dmul(dmul(fx, pu), iz)};
  const double gv[3] = {0.0, dmul(fy, iz), -dmul(dmul(fy, pv), iz)};
  const double col[3][3] = {{0.0, -rx[2], rx[1]}, {rx[2], 0.0, -rx[0]}, {-rx[1], rx[0], 0.0}};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    Jp[0][j] = dot3(gu, col[j]);
    Jp[1][j] = dot3(gv, col[j]);
    Jp[0][3 + j] = gu[j];
    Jp[1][3 + j] = gv[j];
    const double cr[3] = {P[j], P[3 + j], P[6 + j]};
    Jx[0][j] = dot3(gu, cr);
    Jx[1][j] = dot3(gv, cr);
  }
}

// Huber rho(s) for s = |r|^2: s when s <= delta^2, 2 delta sqrt(s) - delta^2 otherwise.
__device__ __forceinline__ double huber_rho(double s, double d, double d2) {
  return s <= d2 ? s : dsub(dmul(dmul(2.0, d), __dsqrt_rn(s)), d2);
}

// Sum of v over the 8 lanes of this lane's track, in ascending frame order (every lane gets the sum).
__device__ __forceinline__ double group_sum(double v) {
  const int base = (threadIdx.x & 31) & ~(MAX_WINDOW - 1);
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < MAX_WINDOW; ++k) s = dadd(s, __shfl_sync(0xffffffffu, v, base + k));
  return s;
}

// Cholesky of the damped 3x3 V (upper: 00 01 02 11 12 22) in lm_solve's order; L lower (00 10 11 20 21 22).
__device__ __forceinline__ bool chol3(const double V[6], double lam, double L[6]) {
  const double a00 = dadd(V[0], dmul(lam, V[0])), a11 = dadd(V[3], dmul(lam, V[3])), a22 = dadd(V[5], dmul(lam, V[5]));
  const double d0 = a00;
  L[0] = __dsqrt_rn(d0);
  L[1] = __ddiv_rn(V[1], L[0]);
  L[3] = __ddiv_rn(V[2], L[0]);
  const double d1 = dsub(a11, dmul(L[1], L[1]));
  L[2] = __dsqrt_rn(d1);
  L[4] = __ddiv_rn(dsub(V[4], dmul(L[3], L[1])), L[2]);
  const double d2 = dsub(dsub(a22, dmul(L[3], L[3])), dmul(L[4], L[4]));
  L[5] = __dsqrt_rn(d2);
  return d0 > 0.0 && d1 > 0.0 && d2 > 0.0;
}

// L y = b.
__device__ __forceinline__ void fwd3(const double L[6], const double b[3], double y[3]) {
  y[0] = __ddiv_rn(b[0], L[0]);
  y[1] = __ddiv_rn(dsub(b[1], dmul(L[1], y[0])), L[2]);
  y[2] = __ddiv_rn(dsub(dsub(b[2], dmul(L[3], y[0])), dmul(L[4], y[1])), L[5]);
}

// L^T x = h.
__device__ __forceinline__ void bwd3(const double L[6], const double h[3], double x[3]) {
  x[2] = __ddiv_rn(h[2], L[5]);
  x[1] = __ddiv_rn(dsub(h[1], dmul(L[4], x[2])), L[2]);
  x[0] = __ddiv_rn(dsub(dsub(h[0], dmul(L[1], x[1])), dmul(L[3], x[2])), L[0]);
}

__device__ __forceinline__ int upper6(int a, int b) { return a * 6 - a * (a - 1) / 2 + (b - a); }

__global__ void __launch_bounds__(GEO_THREADS) ba_kernel(BaParams r) {
  extern __shared__ double stage[];                  // [BA_CHUNK][MAX_WINDOW][SLOT]; S after a forming pass
  __shared__ double sP[2][MAX_WINDOW][12];            // current, candidate pose: R row-major, t
  __shared__ double sU[MAX_WINDOW - 1][SLOT];         // per free frame: U upper (21), b_pose (6)
  __shared__ double sv[MAX_NP], sdp[MAX_NP];          // reduced right-hand side, pose step
  __shared__ double strk[3][BA_CHUNK];                // per-track scalars of a chunk
  __shared__ double s_cost, s_lam, s_sum, s_ntr;
  __shared__ int s_have, s_ok, s_cur;
  const int p = blockIdx.x, tid = threadIdx.x;
  const int c = tid / MAX_WINDOW, w = tid % MAX_WINDOW, gbase = (tid & 31) & ~(MAX_WINDOW - 1);
  const int W = r.W, N = r.N, fixed = r.fixed, nf = W - fixed, NPf = 6 * nf;
  const bool free_w = w >= fixed && w < W;
  const double fx = r.fx, fy = r.fy, cx = r.cx, cy = r.cy, hd = r.huber, hd2 = dmul(r.huber, r.huber);
  const int cnt = min(max(r.counts[p], 0), N);
  double* Xb = reinterpret_cast<double*>(r.ws + (size_t)p * r.ws_window);
  uint8_t* used = r.ws + (size_t)p * r.ws_window + (size_t)N * 6 * sizeof(double);
  const float* pts = r.points + (size_t)p * N * 3;
  const int32_t* ob = r.obs + (size_t)p * N * W;
  int slot = -1;
  if (w < W) slot = r.frame_index[(size_t)p * W + w];

  for (int i = tid; i < W * 12; i += GEO_THREADS)
    sP[0][i / 12][i % 12] = i % 12 < 9 ? r.R[((size_t)p * W + i / 12) * 9 + i % 12]
                                       : r.t[((size_t)p * W + i / 12) * 3 + i % 12 - 9];
  __syncthreads();
  if (tid == 0) {                                      // a non-finite entry or an all-zero R: no model
    bool ok = true;
    for (int f = 0; f < W; ++f) {
      bool nz = false;
      for (int i = 0; i < 12; ++i) ok &= isfinite(sP[0][f][i]);
      for (int i = 0; i < 9; ++i) nz |= sP[0][f][i] != 0.0;
      ok &= nz;
    }
    s_have = ok;
    s_cur = 0;
  }
  __syncthreads();
  const bool have = s_have;

  // keypoint of observation (n, w); false when the index or the slot is out of range or it is not finite
  auto pixel = [&](int n, double& u, double& v) -> bool {
    const int k = ob[(size_t)n * W + w];
    if (slot < 0 || slot >= r.F || k < 0 || k >= r.K) return false;
    const float2 q = reinterpret_cast<const float2*>(r.kpts)[(size_t)slot * r.K + k];
    u = q.x; v = q.y;
    return isfinite(q.x) && isfinite(q.y);
  };
  auto used_obs = [&](int n) { return n < cnt && w < W && ((used[n] >> w) & 1); };
  auto xcur = [&](int n, double X[3]) {
    const double* x = Xb + ((size_t)s_cur * N + n) * 3;
    X[0] = x[0]; X[1] = x[1]; X[2] = x[2];
  };

  // ---- used set, the starting cost and the plain squared error
  double cost0 = 0.0, ss0 = 0.0, nobs = 0.0, ntr = 0.0;          // thread 0's running sums
  if (have) {
    for (int base = 0; base < cnt; base += BA_CHUNK) {
      const int n = base + c;
      bool ok = false;
      double X[3] = {0.0, 0.0, 0.0}, u = 0.0, v = 0.0, s = 0.0, rho = 0.0;
      if (n < cnt) {
        const float* x = pts + (size_t)n * 3;
        X[0] = x[0]; X[1] = x[1]; X[2] = x[2];
        if (w < W && pixel(n, u, v) && isfinite(X[0]) && isfinite(X[1]) && isfinite(X[2]))
          ok = dadd(dot3(sP[0][w] + 6, X), sP[0][w][11]) > 0.0;
      }
      const unsigned bits = (__ballot_sync(0xffffffffu, ok) >> gbase) & 0xffu;
      const bool track = __popc(bits) >= 2;
      if (ok && track) {
        double res[2], z;
        ba_project(sP[0][w], X, u, v, fx, fy, cx, cy, res, z, nullptr, nullptr);
        s = dadd(dmul(res[0], res[0]), dmul(res[1], res[1]));
        rho = huber_rho(s, hd, hd2);
      }
      const double ts = group_sum(s), trho = group_sum(rho);
      if (w == 0 && n < cnt) {
        used[n] = track ? (uint8_t)bits : 0;
        if (track) {
          double* xo = Xb + (size_t)n * 3;
          xo[0] = X[0]; xo[1] = X[1]; xo[2] = X[2];
        }
        strk[0][c] = ts; strk[1][c] = trho; strk[2][c] = track ? __popc(bits) : 0;
      }
      __syncthreads();
      if (tid == 0)
        for (int q = 0; q < BA_CHUNK && base + q < cnt; ++q) {
          ss0 = dadd(ss0, strk[0][q]);
          cost0 = dadd(cost0, strk[1][q]);
          nobs += strk[2][q];
          ntr += strk[2][q] > 0.0 ? 1.0 : 0.0;
        }
      __syncthreads();
    }
  }
  if (tid == 0) { s_cost = cost0; s_ntr = ntr; }
  __syncthreads();
  const bool any_track = s_ntr > 0.0;

  // per-lane linearisation at the current state: weighted Jacobians and residual of a used observation
  auto linearise = [&](int n, double res[2], double wJp[2][6], double Jp[2][6], double wJx[2][3], double Jx[2][3]) {
    double X[3], u = 0.0, v = 0.0, z;
    xcur(n, X);
    pixel(n, u, v);
    ba_project(sP[0][w], X, u, v, fx, fy, cx, cy, res, z, Jp, Jx);
    const double s = dadd(dmul(res[0], res[0]), dmul(res[1], res[1]));
    const double wt = fmin(1.0, __ddiv_rn(hd, __dsqrt_rn(s)));
#pragma unroll
    for (int e = 0; e < 2; ++e) {
#pragma unroll
      for (int i = 0; i < 6; ++i) wJp[e][i] = dmul(wt, Jp[e][i]);
#pragma unroll
      for (int i = 0; i < 3; ++i) wJx[e][i] = dmul(wt, Jx[e][i]);
    }
  };
  // V (6), b_x (3) of the track: the lane's observation's terms summed over the track's frames
  auto point_block = [&](int n, bool use, double V[6], double bx[3]) {
    double Vl[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, bl[3] = {0.0, 0.0, 0.0};
    if (use) {
      double res[2], wJp[2][6], Jp[2][6], wJx[2][3], Jx[2][3];
      linearise(n, res, wJp, Jp, wJx, Jx);
      int q = 0;
      for (int i = 0; i < 3; ++i)
        for (int j = i; j < 3; ++j, ++q) Vl[q] = dadd(dmul(wJx[0][i], Jx[0][j]), dmul(wJx[1][i], Jx[1][j]));
      for (int i = 0; i < 3; ++i) bl[i] = dadd(dmul(wJx[0][i], res[0]), dmul(wJx[1][i], res[1]));
    }
    for (int i = 0; i < 6; ++i) V[i] = group_sum(Vl[i]);
    for (int i = 0; i < 3; ++i) bx[i] = group_sum(bl[i]);
  };
  // Z = W_w L^-T of the lane's (used, free) observation, row a by row a: z(a, Z_a)
  auto z_rows = [&](int n, const double L[6], auto&& z) {
    double res[2], wJp[2][6], Jp[2][6], wJx[2][3], Jx[2][3];
    linearise(n, res, wJp, Jp, wJx, Jx);
    for (int a = 0; a < 6; ++a) {
      const double Wa[3] = {dadd(dmul(wJp[0][a], Jx[0][0]), dmul(wJp[1][a], Jx[1][0])),
                            dadd(dmul(wJp[0][a], Jx[0][1]), dmul(wJp[1][a], Jx[1][1])),
                            dadd(dmul(wJp[0][a], Jx[0][2]), dmul(wJp[1][a], Jx[1][2]))};
      double Za[3];
      fwd3(L, Wa, Za);
      z(a, Za);
    }
  };

  // entries of S (upper, row-major) and of the reduced right-hand side this thread owns
  const int nS = NPf * (NPf + 1) / 2;
  int oi[MAX_OWN], oj[MAX_OWN];
#pragma unroll
  for (int q = 0; q < MAX_OWN; ++q) {
    const int e = tid + q * GEO_THREADS;
    oi[q] = -1; oj[q] = -1;
    if (e < nS) {
      int i = 0, rem = e;
      while (rem >= NPf - i) { rem -= NPf - i; ++i; }
      oi[q] = i; oj[q] = i + rem;
    } else if (e < nS + NPf) {
      oi[q] = e - nS;
    }
  }

  int accepted = 0;
  const bool refine = have && any_track && r.iters > 0;
  bool relin = true;
  for (int it = -1; refine && it < r.iters; ++it) {
    if (relin) {                                       // ---- U, b_pose at the current state (and lambda0)
      double acc = 0.0, dpts = 0.0;
      for (int base = 0; base < cnt; base += BA_CHUNK) {
        const int n = base + c;
        const bool use = used_obs(n);
        double V[6], bx[3], res[2] = {0.0, 0.0}, wJp[2][6], Jp[2][6], wJx[2][3], Jx[2][3];
        point_block(n, use, V, bx);
        if (use && free_w) linearise(n, res, wJp, Jp, wJx, Jx);
        double* st = stage + ((size_t)c * MAX_WINDOW + w) * SLOT;
        int q = 0;
        for (int i = 0; i < 6; ++i)
          for (int j = i; j < 6; ++j, ++q)
            st[q] = use && free_w ? dadd(dmul(wJp[0][i], Jp[0][j]), dmul(wJp[1][i], Jp[1][j])) : 0.0;
        for (int i = 0; i < 6; ++i) st[21 + i] = use && free_w ? dadd(dmul(wJp[0][i], res[0]), dmul(wJp[1][i], res[1])) : 0.0;
        if (w == 0) strk[0][c] = n < cnt && used[n] ? dadd(dadd(V[0], V[3]), V[5]) : 0.0;
        __syncthreads();
        if (tid < nf * SLOT)
          for (int q2 = 0; q2 < BA_CHUNK; ++q2)
            acc = dadd(acc, stage[((size_t)q2 * MAX_WINDOW + fixed + tid / SLOT) * SLOT + tid % SLOT]);
        if (tid == 0)
          for (int q2 = 0; q2 < BA_CHUNK; ++q2) dpts = dadd(dpts, strk[0][q2]);
        __syncthreads();
      }
      if (tid < nf * SLOT) sU[tid / SLOT][tid % SLOT] = acc;
      __syncthreads();
      if (tid == 0 && it < 0) {
        double d = 0.0;
        for (int i = 0; i < NPf; ++i) d = dadd(d, sU[i / 6][upper6(i % 6, i % 6)]);
        d = dadd(d, dpts);
        s_lam = dmul(LM_LAMBDA0, __ddiv_rn(d, (double)NPf + 3.0 * s_ntr));
      }
      __syncthreads();
      relin = false;
      if (it < 0) continue;
    }
    const double lam = s_lam;

    // ---- the reduced camera system S dp = v
    double oacc[MAX_OWN];
#pragma unroll
    for (int q = 0; q < MAX_OWN; ++q) oacc[q] = 0.0;
    bool bad = false;
    for (int base = 0; base < cnt; base += BA_CHUNK) {
      const int n = base + c;
      const bool use = used_obs(n), tr = n < cnt && used[n];
      double V[6], bx[3], L[6], g[3] = {0.0, 0.0, 0.0};
      point_block(n, use, V, bx);
      const bool pd = chol3(V, lam, L);
      bad |= tr && !pd;
      const bool ok = tr && pd;
      if (ok) fwd3(L, bx, g);
      double* st = stage + ((size_t)c * MAX_WINDOW + w) * SLOT;
      if (ok && use && free_w) {
        z_rows(n, L, [&](int a, const double* z) { st[3 * a] = z[0]; st[3 * a + 1] = z[1]; st[3 * a + 2] = z[2]; });
      } else {
        for (int i = 0; i < 18; ++i) st[i] = 0.0;
      }
      st[18] = g[0]; st[19] = g[1]; st[20] = g[2];
      __syncthreads();
#pragma unroll
      for (int q = 0; q < MAX_OWN; ++q) {
        if (oi[q] < 0) continue;
        const int i = oi[q];
        const int fi = fixed + i / 6, ai = i % 6;
        for (int q2 = 0; q2 < BA_CHUNK; ++q2) {
          const double* zi = stage + ((size_t)q2 * MAX_WINDOW + fi) * SLOT + 3 * ai;
          const double* zj = oj[q] >= 0
              ? stage + ((size_t)q2 * MAX_WINDOW + fixed + oj[q] / 6) * SLOT + 3 * (oj[q] % 6)
              : stage + ((size_t)q2 * MAX_WINDOW + fi) * SLOT + 18;
          oacc[q] = dadd(oacc[q], dot3(zi, zj));
        }
      }
      __syncthreads();
    }
    // S = U* - sum Z Z^T into stage (row-major NPf x NPf, lower triangle), v = sum Z g - b_pose
#pragma unroll
    for (int q = 0; q < MAX_OWN; ++q) {
      if (oi[q] < 0) continue;
      const int i = oi[q], j = oj[q];
      if (j >= 0) {
        double u = 0.0;
        if (i / 6 == j / 6) {
          u = sU[i / 6][upper6(i % 6, j % 6)];
          if (i == j) u = dadd(u, dmul(lam, u));
        }
        stage[(size_t)j * NPf + i] = dsub(u, oacc[q]);
      } else {
        sv[i] = dsub(oacc[q], sU[i / 6][21 + i % 6]);
      }
    }
    if (tid == 0) s_ok = 1;
    bad = __syncthreads_or(bad);
    for (int j = 0; j < NPf; ++j) {                     // Cholesky in lm_solve's order
      if (tid == 0) {
        double d = stage[(size_t)j * NPf + j];
        for (int k = 0; k < j; ++k) d = dsub(d, dmul(stage[(size_t)j * NPf + k], stage[(size_t)j * NPf + k]));
        if (!(d > 0.0)) s_ok = 0;
        stage[(size_t)j * NPf + j] = __dsqrt_rn(d);
      }
      __syncthreads();
      for (int i = j + 1 + tid; i < NPf; i += GEO_THREADS) {
        double s = stage[(size_t)i * NPf + j];
        for (int k = 0; k < j; ++k) s = dsub(s, dmul(stage[(size_t)i * NPf + k], stage[(size_t)j * NPf + k]));
        stage[(size_t)i * NPf + j] = __ddiv_rn(s, stage[(size_t)j * NPf + j]);
      }
      __syncthreads();
    }
    if (tid == 0) {
      const double* Lc = stage;
      for (int i = 0; i < NPf; ++i) {
        double s = sv[i];
        for (int k = 0; k < i; ++k) s = dsub(s, dmul(Lc[(size_t)i * NPf + k], sdp[k]));
        sdp[i] = __ddiv_rn(s, Lc[(size_t)i * NPf + i]);
      }
      for (int i = NPf - 1; i >= 0; --i) {
        double s = sdp[i];
        for (int k = i + 1; k < NPf; ++k) s = dsub(s, dmul(Lc[(size_t)k * NPf + i], sdp[k]));
        sdp[i] = __ddiv_rn(s, Lc[(size_t)i * NPf + i]);
      }
      bool fin = true;
      for (int i = 0; i < NPf; ++i) fin &= isfinite(sdp[i]);
      if (!fin) s_ok = 0;
    }
    __syncthreads();
    const bool stepped = s_ok && !bad;
    bool accept = false;
    if (stepped) {
      if (tid < W) {                                    // candidate poses
        double* Pn = sP[1][tid];
        const double* Pc = sP[0][tid];
        if (tid >= fixed) {
          const double* x = sdp + 6 * (tid - fixed);
          double E[9];
          rodrigues(x, E);
          mat3(E, Pc, Pn);
          for (int i = 0; i < 3; ++i) Pn[9 + i] = dadd(Pc[9 + i], x[3 + i]);
        } else {
          for (int i = 0; i < 12; ++i) Pn[i] = Pc[i];
        }
      }
      __syncthreads();
      // ---- back-substitution per track and the candidate's cost
      double costc = 0.0;
      bool behind = false;
      for (int base = 0; base < cnt; base += BA_CHUNK) {
        const int n = base + c;
        const bool use = used_obs(n), tr = n < cnt && used[n];
        double V[6], bx[3], L[6], g[3] = {0.0, 0.0, 0.0};
        point_block(n, use, V, bx);
        chol3(V, lam, L);
        if (tr) fwd3(L, bx, g);
        double ql[3] = {0.0, 0.0, 0.0};
        if (tr && use && free_w) {
          const double* dp = sdp + 6 * (w - fixed);
          z_rows(n, L, [&](int a, const double* z) {
            for (int k = 0; k < 3; ++k) ql[k] = dadd(ql[k], dmul(z[k], dp[a]));
          });
        }
        double h[3], y[3] = {0.0, 0.0, 0.0}, Xc[3] = {0.0, 0.0, 0.0};
        for (int k = 0; k < 3; ++k) h[k] = dadd(g[k], group_sum(ql[k]));
        double rho = 0.0;
        if (tr) {
          bwd3(L, h, y);
          double X[3];
          xcur(n, X);
          for (int k = 0; k < 3; ++k) Xc[k] = dsub(X[k], y[k]);
          if (w == 0) {
            double* xo = Xb + ((size_t)(1 - s_cur) * N + n) * 3;
            xo[0] = Xc[0]; xo[1] = Xc[1]; xo[2] = Xc[2];
          }
        }
        if (use) {
          double u = 0.0, v = 0.0, z, rr[2];
          pixel(n, u, v);
          ba_project(sP[1][w], Xc, u, v, fx, fy, cx, cy, rr, z, nullptr, nullptr);
          behind |= !(z > 0.0);
          rho = huber_rho(dadd(dmul(rr[0], rr[0]), dmul(rr[1], rr[1])), hd, hd2);
        }
        const double trho = group_sum(rho);
        if (w == 0) strk[0][c] = trho;
        __syncthreads();
        if (tid == 0)
          for (int q2 = 0; q2 < BA_CHUNK && base + q2 < cnt; ++q2) costc = dadd(costc, strk[0][q2]);
        __syncthreads();
      }
      behind = __syncthreads_or(behind);
      if (tid == 0) s_sum = costc;
      __syncthreads();
      accept = !behind && s_sum < s_cost;
    }
    if (accept) {
      if (tid < W * 12) sP[0][tid / 12][tid % 12] = sP[1][tid / 12][tid % 12];
      __syncthreads();
      if (tid == 0) {
        s_cur = 1 - s_cur;
        s_cost = s_sum;
        s_lam = __ddiv_rn(s_lam, LM_LAMBDA_STEP);
      }
      ++accepted;
    } else if (tid == 0) {
      s_lam = dmul(s_lam, LM_LAMBDA_STEP);
    }
    __syncthreads();
    relin = accept && it + 1 < r.iters;
  }

  // ---- outputs: poses, points, the final mask and squared error
  double ss1 = 0.0;
  for (int base = 0; base < N; base += BA_CHUNK) {
    const int n = base + c;
    const bool use = have && used_obs(n), tr = have && n < cnt && used[n];
    double s = 0.0;
    double X[3] = {0.0, 0.0, 0.0};
    if (tr) xcur(n, X);
    if (use) {
      double u = 0.0, v = 0.0, z, rr[2];
      pixel(n, u, v);
      ba_project(sP[0][w], X, u, v, fx, fy, cx, cy, rr, z, nullptr, nullptr);
      s = dadd(dmul(rr[0], rr[0]), dmul(rr[1], rr[1]));
    }
    const double ts = group_sum(s);
    if (n < N) {
      if (r.mask && w < W) r.mask[((size_t)p * N + n) * W + w] = use && s < r.t2;
      if (w < 3) {
        float* o = r.points_out + ((size_t)p * N + n) * 3;
        o[w] = tr ? __double2float_rn(X[w]) : pts[(size_t)n * 3 + w];
      }
    }
    if (w == 0) strk[0][c] = ts;
    __syncthreads();
    if (tid == 0)
      for (int q2 = 0; q2 < BA_CHUNK && base + q2 < cnt; ++q2) ss1 = dadd(ss1, strk[0][q2]);
    __syncthreads();
  }
  for (int i = tid; i < W * 12; i += GEO_THREADS) {
    const int f = i / 12, e = i % 12;
    if (e < 9) r.R_out[((size_t)p * W + f) * 9 + e] = sP[0][f][e];
    else r.t_out[((size_t)p * W + f) * 3 + e - 9] = sP[0][f][e];
  }
  if (tid == 0) {
    const bool any = have && nobs > 0.0;
    r.rms[2 * (size_t)p] = any ? __dsqrt_rn(__ddiv_rn(ss0, nobs)) : 0.0;
    r.rms[2 * (size_t)p + 1] = any ? __dsqrt_rn(__ddiv_rn(ss1, nobs)) : 0.0;
    if (r.accepted) r.accepted[p] = accepted;
  }
}

}  // namespace
}  // namespace sslam

using namespace sslam;

extern "C" size_t sslam_bundle_adjust_workspace_bytes(int P, int N) {
  return P > 0 && N >= 0 ? (size_t)P * ws_window_bytes(N) : 0;
}

extern "C" int sslam_bundle_adjust(const float* kpts, int F, int K, const int32_t* frame_index, int P, int W, int N,
                                   const int32_t* obs, const float* points, const int32_t* counts, const double* R,
                                   const double* t, double fx, double fy, double cx, double cy, int fixed,
                                   double huber, double threshold, int refine_iters, double* R_out, double* t_out,
                                   float* points_out, double* rms, int32_t* accepted, uint8_t* mask, void* ws,
                                   size_t ws_bytes, void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  SSLAM_REQUIRE(W <= MAX_WINDOW, SSLAM_EUNSUPPORTED, "bundle_adjust: window of %d frames > %d", W, MAX_WINDOW);
  SSLAM_REQUIRE(W >= 2, SSLAM_EINVAL, "bundle_adjust: a window needs at least 2 frames (W=%d)", W);
  SSLAM_REQUIRE(N <= MAX_TRACKS, SSLAM_EUNSUPPORTED, "bundle_adjust: %d tracks > %d", N, MAX_TRACKS);
  SSLAM_REQUIRE(fixed >= 1 && fixed <= W, SSLAM_EINVAL, "bundle_adjust: fixed=%d (need 1..%d)", fixed, W);
  SSLAM_REQUIRE(huber > 0.0 && !isnan(huber), SSLAM_EINVAL, "bundle_adjust: huber must be > 0 (inf: none)");
  const double Kc[4] = {fx, fy, cx, cy};
  rc = check_list_args("bundle_adjust", P, N, K, 0, F, F, frame_index,
                       kpts && frame_index && obs && points && counts && R && t && R_out && t_out && points_out &&
                           rms && ws,
                       nullptr, &refine_iters, "threshold", threshold, Kc);
  if (rc || P == 0) return rc;
  const size_t need = sslam_bundle_adjust_workspace_bytes(P, N);
  SSLAM_REQUIRE(ws_bytes >= need, SSLAM_EWORKSPACE, "bundle_adjust: workspace %zu B < %zu B", ws_bytes, need);
  static DeviceOnce once;
  if (once.first_use())
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(ba_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STAGE_BYTES));
  cudaStream_t stream = (cudaStream_t)stream_;
  BaParams r{kpts, F, K, frame_index, P, W, N, obs, points, counts, R, t, fx, fy, cx, cy, huber,
             threshold * threshold, fixed, refine_iters, R_out, t_out, points_out, rms, accepted, mask,
             (uint8_t*)ws, ws_window_bytes(N)};
  SSLAM_LAUNCH(KK_BUNDLE_ADJUST, stream, ba_kernel<<<P, GEO_THREADS, STAGE_BYTES, stream>>>(r));
  return SSLAM_OK;
}
