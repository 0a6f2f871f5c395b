// Shared device/host helpers for libsslam_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>

#include "../../include/sslam_b200.h"

namespace sslam {

typedef unsigned long long u64;
typedef unsigned int u32;

// ---------------------------------------------------------------------------- host side
void set_error(const char* fmt, ...);
int check_device();                    // cached per device; SSLAM_OK or error
int num_sms();                         // of the calling thread's current device
// True exactly once per (call site, device): function attributes (dynamic shared memory size) and
// occupancy answers are per device, so a process that drives several GPUs configures each of them.
//   static DeviceOnce once;  if (once.first_use()) { cudaFuncSetAttribute(...); }
struct DeviceOnce {
  std::atomic<uint64_t> done[2] = {};
  bool first_use() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return true;
    const uint64_t bit = 1ull << (dev & 63);
    std::atomic<uint64_t>& w = done[(dev >> 6) & 1];
    if (w.load(std::memory_order_acquire) & bit) return false;
    w.fetch_or(bit, std::memory_order_acq_rel);
    return true;
  }
};
extern std::atomic<uint64_t> g_launches;

#define SSLAM_CHECK_CUDA(expr)                                                        \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      ::sslam::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                         __FILE__, __LINE__);                                         \
      return SSLAM_ECUDA;                                                             \
    }                                                                                 \
  } while (0)

#define SSLAM_REQUIRE(cond, code, ...)                                                \
  do {                                                                                \
    if (!(cond)) {                                                                    \
      ::sslam::set_error(__VA_ARGS__);                                                \
      return (code);                                                                  \
    }                                                                                 \
  } while (0)

// kernel kinds for the launch counter / optional per-kernel event timing (sslam_profile_*)
enum KernelKind {
  KK_DECODE_SCAN = 0, KK_DECODE_TOPK, KK_DECODE_COUNT, KK_DECODE_RESOLVE, KK_NMS, KK_GATHER, KK_L2NORM,
  KK_MATCH_F32, KK_MATCH_TC, KK_SPLIT, KK_UNPACK, KK_FINALIZE, KK_GEMM, KK_LAYERNORM, KK_EVAL, KK_HEATMAP,
  KK_CONV_HEAD, KK_RANSAC_HYP, KK_RANSAC_SCORE, KK_RANSAC_REFIT, KK_COUNT
};
extern std::atomic<int> g_profile_on;
void prof_mark(int kind, cudaStream_t stream, bool begin);

// SSLAM_LAUNCH(kind, stream, kernel<<<grid, block, smem, stream>>>(args...));
#define SSLAM_LAUNCH(kind, stream, ...)                                               \
  do {                                                                                \
    if (::sslam::g_profile_on.load(std::memory_order_relaxed))                        \
      ::sslam::prof_mark(kind, stream, true);                                         \
    __VA_ARGS__;                                                                      \
    if (::sslam::g_profile_on.load(std::memory_order_relaxed))                        \
      ::sslam::prof_mark(kind, stream, false);                                        \
    ::sslam::g_launches.fetch_add(1, std::memory_order_relaxed);                      \
    SSLAM_CHECK_CUDA(cudaGetLastError());                                             \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------- device side
#ifdef __CUDACC__

// order-preserving map fp32 -> u32 (works for negatives; NaNs sort to the extremes)
__device__ __forceinline__ u32 ordered_from_float(float f) {
  u32 b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float float_from_ordered(u32 o) {
  u32 b = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  return __uint_as_float(b);
}
// key whose max is (largest value, lowest index)
__device__ __forceinline__ u64 pack_key(float v, u32 idx) {
  return ((u64)ordered_from_float(v) << 32) | (u64)(0xffffffffu - idx);
}
__device__ __forceinline__ float key_value(u64 k) { return float_from_ordered((u32)(k >> 32)); }
__device__ __forceinline__ u32 key_index(u64 k) { return 0xffffffffu - (u32)(k & 0xffffffffu); }

__device__ __forceinline__ float sigmoid_f32(float x) { return 1.0f / (1.0f + expf(-x)); }

// ATen CPU lerp as used by torch.quantile: one FMA (see oracle/decode.py::quantile_f32)
__device__ __forceinline__ float lerp_aten(float a, float b, float w) {
  float d = __fsub_rn(b, a);
  return (fabsf(w) < 0.5f) ? __fmaf_rn(w, d, a) : __fmaf_rn(__fsub_rn(w, 1.0f), d, b);
}

template <typename T>
__device__ __forceinline__ T warp_reduce_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum for blockDim.x <= 1024 (multiple of 32). `red` is >= 33 elements of smem.
template <typename T>
__device__ __forceinline__ T block_reduce_sum(T v, T* red) {
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_reduce_sum(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    T t = (lane < nw) ? red[lane] : T(0);
    t = warp_reduce_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

// ----------------------------------------------------------------------------
// Exact k-th largest of a (filtered) key stream, whole block cooperates.
//
// `src(i, key)` returns false when element i is not part of the set.  Keys need not be distinct.
// MSB-first radix select, but each round first finds the highest bit in which the still-active
// keys differ and places an 11-bit digit there, so runs of identical high bits (all scores in
// [0.5,1) share sign+exponent) cost nothing and histograms are spread over the bins.
// Returns the r-th largest key (r is 1-based, 1 <= r <= active count).
struct SelectScratch {
  u32 hist[2048];
  u64 or_and[2];
  u64 red_or[32];
  u64 red_and[32];
  u32 pick_bin;
  u32 pick_rank;
  u32 lane_sum[32];
};

template <typename Src>
__device__ u64 block_select_kth_largest(Src src, int n, u32 r, SelectScratch* s) {
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = nth >> 5;
  u64 mask = 0, val = 0;  // bits already decided
  for (;;) {
    // ---- pass 1: OR / AND of active keys
    u64 o = 0, a = ~0ull;
    for (int i = tid; i < n; i += nth) {
      u64 k;
      if (src(i, k) && (k & mask) == val) { o |= k; a &= k; }
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
      o |= __shfl_xor_sync(0xffffffffu, o, sft);
      a &= __shfl_xor_sync(0xffffffffu, a, sft);
    }
    __syncthreads();
    if (lane == 0) { s->red_or[warp] = o; s->red_and[warp] = a; }
    __syncthreads();
    if (tid == 0) {
      u64 oo = 0, aa = ~0ull;
      for (int w = 0; w < nwarps; ++w) { oo |= s->red_or[w]; aa &= s->red_and[w]; }
      s->or_and[0] = oo; s->or_and[1] = aa;
    }
    for (int i = tid; i < 2048; i += nth) s->hist[i] = 0;
    __syncthreads();
    o = s->or_and[0]; a = s->or_and[1];
    u64 diff = (o ^ a) & ~mask;
    if (diff == 0) return o;                      // every active key is identical
    int hb = 63 - __clzll((long long)diff);       // highest differing bit
    int shift = hb - 10; if (shift < 0) shift = 0;
    // bits above the digit window that are not yet decided are common to all active keys
    u64 above = ~((hb >= 63) ? ~0ull : ((1ull << (hb + 1)) - 1));
    val |= (a & above & ~mask); mask |= above;
    // ---- pass 2: histogram of the digit
    for (int i = tid; i < n; i += nth) {
      u64 k;
      if (src(i, k) && (k & mask) == val) atomicAdd(&s->hist[(u32)(k >> shift) & 2047u], 1u);
    }
    __syncthreads();
    // ---- locate the bin holding the r-th largest (scan from the top bin down); warp 0
    if (warp == 0) {
      // lane L owns bins [2047-64L-63 .. 2047-64L] i.e. descending order by lane
      u32 sum = 0;
      int top = 2047 - 64 * lane;
      for (int b = 0; b < 64; ++b) sum += s->hist[top - b];
      u32 incl = sum;
#pragma unroll
      for (int sft = 1; sft < 32; sft <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, incl, sft);
        if (lane >= sft) incl += t;
      }
      u32 excl = incl - sum;
      if (r > excl && r <= incl) {                // exactly one lane
        u32 need = r - excl, c = 0;
        for (int b = 0; b < 64; ++b) {
          u32 h = s->hist[top - b];
          if (c + h >= need) { s->pick_bin = (u32)(top - b); s->pick_rank = need - c; break; }
          c += h;
        }
      }
    }
    __syncthreads();
    u32 bin = s->pick_bin;
    r = s->pick_rank;
    u64 digit_mask = 2047ull << shift;
    val |= ((u64)bin << shift) & digit_mask;
    mask |= digit_mask;
    __syncthreads();
    if (shift == 0) return val;                   // all 64 bits decided
  }
}

// In-place bitonic sort, descending, of `n_pow2` u64 keys in shared memory.
__device__ __forceinline__ void block_bitonic_sort_desc(u64* keys, int n_pow2) {
  const int tid = threadIdx.x, nth = blockDim.x;
  for (int k = 2; k <= n_pow2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int t = tid; t < (n_pow2 >> 1); t += nth) {
        int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));   // index with bit j clear
        int p = i | j;
        bool desc = ((i & k) == 0);
        u64 x = keys[i], y = keys[p];
        if ((x < y) == desc) { keys[i] = y; keys[p] = x; }
      }
    }
  }
  __syncthreads();
}

#endif  // __CUDACC__
}  // namespace sslam
