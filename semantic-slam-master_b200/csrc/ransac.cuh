// The three-launch RANSAC shared by the homography and fundamental matrix (ransac.cu) and the PnP
// (pnp.cu) estimators, as templates over the model M:
//
//   ransac_hyp     one thread per (list, sample): M::SAMPLE distinct rows drawn by the splitmix64
//                  sampler, M::solve -> M::SLOTS hypotheses of M::FLOATS floats each
//   ransac_score   the hot loop (P x SLOTS*iters x n inlier tests): the list's rows are staged in shared
//                  memory tile by tile (M::TILE rows of M::ROW_FLOATS floats), warps take hypotheses,
//                  lanes stride the rows
//   refit          one CTA per list, a kernel of each estimator built from best_keys / best_slot,
//                  mask_pass, keep_refit and finish_lists below
//
// A model M provides SAMPLE, SLOTS, FLOATS, TILE, ROW_FLOATS; Row and row(r, p, a, b, k), the list's row k
// (NaN where an index is out of range); solve(q, r, H), the minimal solve from the drawn rows q, bit k of
// its result set when slot k holds a model; inlier(h, row, r); and stage(s, tile, k, row) /
// staged(s, tile, k), how a row is written to and read from the score tile s.
#pragma once

#include "geometry.cuh"

namespace sslam {
namespace {

constexpr int HYP_THREADS = 64;
constexpr int SC_THREADS = 256;
constexpr int SC_HYPS = 256;          // hypotheses per scoring CTA (32 per warp)

struct RansacParams {
  const float* k1; const float* k2;          // [F1,N,2] ([F1,N,3] points for PnP), [F2,M,2]
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
  float* hyp;                                // [P,SLOTS*iters,FLOATS]
  // PnP only (after the shared fields, so that their offsets do not depend on the model)
  double fx, fy, cx, cy;
  int refine_iters;
  double* R; double* t; double* rms;         // [P,9], [P,3], [P,2] or null
};

// Slots of sample s of list p as doubles: bit k set when slot k holds a model.
template <class M>
__device__ __forceinline__ int sample_hyps(const RansacParams& r, int p, int a, int b, int n, int s,
                                           double Hs[M::SLOTS][M::FLOATS]) {
  int idx[M::SAMPLE];
#pragma unroll
  for (int k = 0; k < M::SAMPLE; ++k) idx[k] = -1;
  if (n < M::SAMPLE || !sample_rows<M::SAMPLE>(r.seed, s, n, idx)) return 0;
  typename M::Row q[M::SAMPLE];
#pragma unroll
  for (int k = 0; k < M::SAMPLE; ++k) q[k] = M::row(r, p, a, b, idx[k]);
  return M::solve(q, r, Hs);
}

template <class M>
__global__ void __launch_bounds__(HYP_THREADS) ransac_hyp_kernel(RansacParams r) {
  const int p = blockIdx.x;
  const int s = blockIdx.y * HYP_THREADS + threadIdx.x;
  if (s >= r.iters) return;
  int a, b;
  const int n = pair_rows(r, p, a, b);
  double H[M::SLOTS][M::FLOATS];
  const int ok = sample_hyps<M>(r, p, a, b, n, s, H);
#pragma unroll
  for (int j = 0; j < M::SLOTS; ++j) {
    const size_t h = ((size_t)p * r.iters + s) * M::SLOTS + j;
    const bool v = (ok >> j) & 1;
    float* o = r.hyp + h * M::FLOATS;
#pragma unroll
    for (int k = 0; k < M::FLOATS; ++k) o[k] = v ? __double2float_rn(H[j][k]) : 0.f;
    r.hyp_count[h] = v ? 0 : -1;
  }
}

template <class M>
__global__ void __launch_bounds__(SC_THREADS) ransac_score_kernel(RansacParams r, int tile) {
  extern __shared__ float4 stage_mem[];              // tile rows of M::ROW_FLOATS floats
  float* rows = reinterpret_cast<float*>(stage_mem);
  __shared__ float hs[SC_HYPS][M::FLOATS];
  __shared__ int cnt[SC_HYPS];
  const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slots = M::SLOTS * r.iters;
  const int h0 = blockIdx.y * SC_HYPS;
  const int nh = min(SC_HYPS, slots - h0);
  int a, b;
  const int n = pair_rows(r, p, a, b);
  if (n < M::SAMPLE) return;                           // every hypothesis of the list is degenerate
  const size_t base = (size_t)p * slots + h0;
  for (int t = tid; t < nh * M::FLOATS; t += SC_THREADS)
    hs[t / M::FLOATS][t % M::FLOATS] = r.hyp[base * M::FLOATS + t];
  for (int t = tid; t < nh; t += SC_THREADS) cnt[t] = r.hyp_count[base + t];
  for (int k0 = 0; k0 < n; k0 += tile) {
    const int nt = min(tile, n - k0);
    __syncthreads();
    for (int k = tid; k < nt; k += SC_THREADS) M::stage(rows, tile, k, M::row(r, p, a, b, k0 + k));
    __syncthreads();
    for (int hl = warp; hl < nh; hl += SC_THREADS / 32) {
      if (cnt[hl] < 0) continue;
      float h[M::FLOATS];
#pragma unroll
      for (int k = 0; k < M::FLOATS; ++k) h[k] = hs[hl][k];
      int c = 0;
      for (int k0 = 0; k0 < nt; k0 += 32) {              // warp-uniform bound: every lane votes
        const int k = k0 + lane;
        c += __popc(__ballot_sync(0xffffffffu, k < nt && M::inlier(h, M::staged(rows, tile, k), r)));
      }
      if (lane == 0) cnt[hl] += c;
    }
  }
  __syncthreads();
  for (int t = tid; t < nh; t += SC_THREADS) r.hyp_count[base + t] = cnt[t];
}

// ---------------------------------------------------------------------------- refit pieces
// Every thread of the refit CTA (GEO_THREADS) calls these.

// Best slot of list p: most inliers, lowest slot on ties, as the largest key (count + 1, ~slot); every
// thread calls best_keys, which leaves each warp's best key in bkey (shared [GEO_THREADS / 32]), then
// thread 0 calls best_slot: the slot, or -1 when no slot holds a model.
template <class M>
__device__ __forceinline__ void best_keys(const RansacParams& r, int p, int n, unsigned long long* bkey) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slots = M::SLOTS * r.iters;
  unsigned long long key = 0;
  if (n >= M::SAMPLE)
    for (int h = tid; h < slots; h += GEO_THREADS) {
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
}

__device__ __forceinline__ int best_slot(const unsigned long long* bkey) {
  unsigned long long k = 0;
  for (int w = 0; w < GEO_THREADS / 32; ++w) k = bkey[w] > k ? bkey[w] : k;
  return (k >> 32) == 0 ? -1 : (int)(0xffffffffu - (unsigned)(k & 0xffffffffu));
}

// Inliers of the best hypothesis hf (none when !have) into flag[] and the workspace's hyp_mask; returns
// their number.  scan: shared [GEO_THREADS], the reduction scratch.
template <class M>
__device__ __forceinline__ int mask_pass(const RansacParams& r, int p, int a, int b, int n, bool have,
                                         const float* hf, uint8_t* flag, int* scan) {
  uint8_t* hm = r.hyp_mask + (size_t)p * r.L;
  int m = 0;
  for (int k = threadIdx.x; k < r.L; k += GEO_THREADS) {
    const bool in = have && k < n && M::inlier(hf, M::row(r, p, a, b, k), r);
    flag[k] = in;
    hm[k] = in;
    m += in;
  }
  return block_reduce_sum(m, scan);
}

// Whether the refit hf is kept: it has at least as many inliers as the best hypothesis's m.
template <class M>
__device__ __forceinline__ bool keep_refit(const RansacParams& r, int p, int a, int b, int n, const float* hf,
                                           int m, int* scan) {
  int c = 0;
  for (int k = threadIdx.x; k < n; k += GEO_THREADS) c += M::inlier(hf, M::row(r, p, a, b, k), r);
  c = block_reduce_sum(c, scan);
  return c >= m;
}

// Order-preserving compaction of the kept rows flag[] into the matcher's list format, the mask and the
// count.  s_total: shared.
__device__ __forceinline__ void finish_lists(const RansacParams& r, int p, int n, const uint8_t* flag, int* scan,
                                             int* s_total) {
  const int tid = threadIdx.x;
  __syncthreads();
  const int total = compact_rows(flag, n, r.L, p, r.pairs, r.pair_scores, r.out_pairs, r.out_scores, scan, s_total);
  if (r.mask)
    for (int k = tid; k < r.L; k += GEO_THREADS) r.mask[(size_t)p * r.L + k] = k < n ? flag[k] : 0;
  if (tid == 0) r.out_counts[p] = total;
}

// ---------------------------------------------------------------------------- host side
template <class M>
size_t ransac_workspace_bytes(int P, int L, int iters) {
  if (P <= 0 || L < 0 || iters <= 0) return 0;
  return ws_layout(P, L, iters, M::SLOTS, M::FLOATS).total;
}

// Carves the workspace into r and launches the three kernels of model M (profiled as kinds[0..2]);
// arguments checked by check_list_args, P > 0.
template <class M>
int ransac_launch(const char* fn, RansacParams& r, void* ws, size_t ws_bytes, void (*refit)(RansacParams),
                  const int (&kinds)[3], cudaStream_t stream) {
  const WsLayout w = ws_layout(r.P, r.L, r.iters, M::SLOTS, M::FLOATS);
  SSLAM_REQUIRE(ws_bytes >= w.total, SSLAM_EWORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, w.total);
  char* base = static_cast<char*>(ws);
  r.hyp_count = reinterpret_cast<int32_t*>(base + w.count);
  r.best = reinterpret_cast<int32_t*>(base + w.best);
  r.hyp_mask = reinterpret_cast<uint8_t*>(base + w.mask);
  r.hyp = reinterpret_cast<float*>(base + w.hyp);
  const int tile = r.L < 1 ? 1 : (r.L < M::TILE ? r.L : M::TILE);
  const size_t smem = (size_t)tile * M::ROW_FLOATS * sizeof(float);
  const int score_ctas = (M::SLOTS * r.iters + SC_HYPS - 1) / SC_HYPS;
  static DeviceOnce once;
  if (once.first_use())
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(ransac_score_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(M::TILE * M::ROW_FLOATS * sizeof(float))));
  SSLAM_LAUNCH(kinds[0], stream,
               ransac_hyp_kernel<M><<<dim3(r.P, (r.iters + HYP_THREADS - 1) / HYP_THREADS), HYP_THREADS, 0,
                                      stream>>>(r));
  SSLAM_LAUNCH(kinds[1], stream, ransac_score_kernel<M><<<dim3(r.P, score_ctas), SC_THREADS, smem, stream>>>(r, tile));
  SSLAM_LAUNCH(kinds[2], stream, refit<<<r.P, GEO_THREADS, 0, stream>>>(r));
  return SSLAM_OK;
}

}  // namespace
}  // namespace sslam
