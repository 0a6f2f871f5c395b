// DescriptorRefiner forward on tensor cores (SURVEY.md §8(f) N1).
//
// Replaces the body of DescriptorRefiner.forward / ResidualBlock.forward
// (models/descriptor_refiner.py:73-86, 108-126): Linear+ReLU, [LN, Linear+ReLU, LN, Linear,
// +identity, ReLU] x blocks, Linear, L2 normalise — with fp32-level accuracy at the full 16-bit
// tensor-core rate:
//
//   * numbers are carried as fp16 PAIRS, x ~= hi + lo * 2^-11 (hi = fp16(x), lo = fp16((x-hi) * 2^11):
//     22 significant bits), and every Linear is three tcgen05 kind::f16 MMAs
//         x.w ~= hi.hi'  +  2^-11 * (hi.lo' + lo.hi')
//     with fp32 accumulation in TMEM; the cross terms live in their own accumulator and are folded
//     in by the epilogue with one FMA (the tensor core truncates when it adds into an accumulator,
//     so small terms must not be added to a large one inside it).  The dropped lo.lo' term is 2^-22.
//   * activations travel between layers as such pairs (two fp16 arrays = 4 bytes per element, the
//     same HBM traffic as fp32) and are loaded by TMA straight into 128B-swizzled operand tiles —
//     no conversion stage, no fp32 activations in HBM; weights are split once by
//     sslam_refiner_pack_weights.  Requires |activation| < 65504.
//   * the GEMM epilogue (thread = row, tcgen05.ld, 16 columns at a time) fuses bias / folded
//     LayerNorm, residual add, ReLU and the row statistics, packs the next layer's pair (or fp32 for
//     the last layer) into a dense shared-memory box and hands it to a TMA store, which also clips
//     ragged rows / columns; no per-lane global stores.
//   * LayerNorm never runs as a kernel.  For y = LN(h).W^T + c with LN(h) = (h - mu) * rho * g + b,
//         y[r,n] = rho_r * ( (h.W'^T)[r,n] - mu_r * s1[n] ) + c0[n],
//     W' = W * g (column scale), s1[n] = sum_k W'[n,k], c0[n] = sum_k b[k] W[n,k] + c[n]  (all folded
//     once by sslam_refiner_pack_weights).  So the GEMM multiplies the *un-normalised* activations
//     and its epilogue applies the two per-row scalars; those (mu_r, rho_r) are produced for free by
//     the epilogue of the GEMM that wrote h (row sums of v and v^2 while storing).
//
// Three kernels.  refiner_fused_kernel (last in this file) is the production path for C, Hd <= 384:
// ONE persistent launch for all layers, weight-stationary CTA pairs (cta_group::2, M = 256) in clusters
// that multicast the activation blocks, activations exchanged between layers through an L2-resident
// scratch in the UMMA operand layout.  gemm_pair_kernel is the same data path with one launch per layer
// (fallback, and the bit-exact cross-check of the fused kernel); gemm_f16x3_kernel (directly below) is
// the general single-CTA fallback: persistent, one CTA per SM, each CTA walks 128-row strips and,
// inside a strip, the N/128 column tiles of the layer, streaming both operands.
#include "tc_common.cuh"

namespace sslam {

using namespace tc;

// sticky range flag of the fp16-pair arithmetic (sslam_refiner_range_check); one copy per device
__device__ unsigned int g_refiner_status = 0;
constexpr float F16_RANGE_SQ = 65504.0f * 65504.0f;

int g_refiner_fused = 3;            // 0: one launch per layer; 1..4: layer-fused kernel, strip pairs per chunk (sslam_debug_refiner_fused)

namespace {

constexpr int BM = 128, BN = 128, BK = 64;               // BK fp16 = 128 bytes of K
constexpr int BLOCK_BYTES = BM * 128;
constexpr int STAGES = 3;
constexpr int STAGE_BYTES = 4 * BLOCK_BYTES;             // A_hi, A_lo, B_hi, B_lo
constexpr int EPI_WARPS = 8;                             // two warps per TMEM lane quarter
constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
constexpr int TMEM_COLS = 512;                           // 2 x (128 main + 128 cross)
constexpr int UNIT = 16;                                 // columns per epilogue step
constexpr int STG_BYTES = 32 * UNIT * 4;                 // per warp: [32][16] fp16 hi | lo, or [32][16] fp32
constexpr int SMEM_OPERANDS = STAGES * STAGE_BYTES;
constexpr int SMEM_TRANSP = EPI_WARPS * STG_BYTES;
constexpr int SMEM_STATS = 2 * 4 * 32 * 2 * 2 * 4;         // [parity][quarter][row][half][sum, sumsq]
constexpr int MAX_N = 1024;
constexpr int SMEM_VECS = 2 * MAX_N * 4;                 // bias / c0 and s1 of the layer, staged once per CTA
constexpr int SMEM_BARS = (2 * STAGES + 4) * 8 + 16;
constexpr int SMEM_TOTAL = SMEM_OPERANDS + SMEM_TRANSP + SMEM_STATS + SMEM_VECS + SMEM_BARS + 1024;

struct GemmParams {
  int rows, N, K;
  const float* bias;        // [N]
  const __half* res_hi;     // residual pair [rows, N] or null
  const __half* res_lo;
  int relu;
  float* out_f32;           // [rows, N] or null
  __half* out_hi;           // pair [rows, N] or null
  __half* out_lo;
  // folded LayerNorm on the A operand (null = plain bias): partial row sums / sums of squares of A
  // ([a_parts][stat_stride], written by the GEMM that produced A), per-column s1; `bias` then holds c0
  const float* a_sum;
  const float* a_sq;
  int a_parts;
  const float* s1;
  // partial row sums of the OUTPUT (after residual + ReLU) for the next folded LayerNorm, or null:
  // part = column tile of the writer (pair kernel) or 0 (single-CTA kernel)
  float* out_sum;
  float* out_sq;
  size_t stat_stride;
};

// 32 contiguous, 32-byte aligned bytes through the read-only path as one 256-bit load
__device__ __forceinline__ void ldg_256(const void* ptr, uint4 (&d)[2]) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(d[0].x), "=r"(d[0].y), "=r"(d[0].z), "=r"(d[0].w), "=r"(d[1].x), "=r"(d[1].y), "=r"(d[1].z),
                 "=r"(d[1].w)
               : "l"(ptr));
}

// mean / rstd of row `grow` of the A operand from the producer's partial sums (fixed summation order)
__device__ __forceinline__ void row_layernorm_scalars(const GemmParams& p, int grow, float& mean, float& rstd) {
  float sm = 0.f, sq = 0.f;
  for (int i = 0; i < p.a_parts; ++i) {
    sm += __ldg(p.a_sum + (size_t)i * p.stat_stride + grow);
    sq += __ldg(p.a_sq + (size_t)i * p.stat_stride + grow);
  }
  mean = sm / (float)p.K;
  const float var = fmaxf(sq / (float)p.K - mean * mean, 0.f);
  rstd = 1.0f / sqrtf(var + 1e-5f);
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_f16x3_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                  const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                  const __grid_constant__ CUtensorMap tmO_hi, const __grid_constant__ CUtensorMap tmO_lo,
                  const __grid_constant__ CUtensorMap tmO_f32, GemmParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* operands = smem;
  unsigned char* staging = smem + SMEM_OPERANDS;
  float* stats = reinterpret_cast<float*>(smem + SMEM_OPERANDS + SMEM_TRANSP);
  float* sbias = reinterpret_cast<float*>(smem + SMEM_OPERANDS + SMEM_TRANSP + SMEM_STATS);
  float* ss1 = sbias + MAX_N;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SMEM_OPERANDS + SMEM_TRANSP + SMEM_STATS + SMEM_VECS);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nstrips = (p.rows + BM - 1) / BM;       // persistent: strips blockIdx.x, +gridDim.x, ...
  const int ntile = (p.N + BN - 1) / BN;
  const int nkb = (p.K + BK - 1) / BK;
  // Every CTA multiplies by the same weight matrix; walking its tiles in lock-step would make all
  // 148 SMs hit the same few L2 lines at once.  Each CTA therefore starts at its own column tile
  // and its own k-block (the k order only changes the fp32 summation order).
  const int ct_rot = blockIdx.x % ntile;
  const int kb_rot = (blockIdx.x / ntile) % nkb;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  for (int i = threadIdx.x; i < p.N; i += NUM_THREADS) {        // per-column vectors -> smem
    sbias[i] = __ldg(p.bias + i);
    ss1[i] = p.a_sum ? __ldg(p.s1 + i) : 0.f;
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {                                            // ---- TMA producer
      prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmA_lo);
      prefetch_tensormap(&tmB_hi); prefetch_tensormap(&tmB_lo);
      int stage = 0; uint32_t phase = 0;
      for (int strip = blockIdx.x; strip < nstrips; strip += gridDim.x) {
        const int row0 = strip * BM;
        for (int ct = 0; ct < ntile; ++ct) {
          for (int kb = 0; kb < nkb; ++kb) {
            mbar_wait(&empty[stage], phase ^ 1);
            unsigned char* st = operands + stage * STAGE_BYTES;
            mbar_arrive_expect_tx(&full[stage], STAGE_BYTES);
            int kr = kb + kb_rot; if (kr >= nkb) kr -= nkb;
            int cr = ct + ct_rot; if (cr >= ntile) cr -= ntile;
            const int kc = kr * BK;
            tma_load_2d(st, &tmA_hi, &full[stage], kc, row0);
            tma_load_2d(st + BLOCK_BYTES, &tmA_lo, &full[stage], kc, row0);
            tma_load_2d(st + 2 * BLOCK_BYTES, &tmB_hi, &full[stage], kc, cr * BN);
            tma_load_2d(st + 3 * BLOCK_BYTES, &tmB_lo, &full[stage], kc, cr * BN);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {                                            // ---- MMA issuer
      const uint32_t idesc = make_instr_desc(FMT_F16, BM, BN);
      const uint32_t idesc_cat = make_instr_desc(FMT_F16, BM, 2 * BN);
      int stage = 0; uint32_t phase = 0;
      const int my_tiles = ((nstrips - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x) * ntile;
      for (int tc = 0; tc < my_tiles; ++tc) {           // tc: running tile count of this CTA
        const int acc = tc & 1;
        mbar_wait(&tempty[acc], ((tc >> 1) & 1) ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * 2 * BN;
        const uint32_t tmem_s = tmem_d + BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full[stage], phase);               // TMA bytes have landed
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(operands + stage * STAGE_BYTES);
          const uint64_t a_hi = make_smem_desc_sw128(sa);
          const uint64_t a_lo = make_smem_desc_sw128(sa + BLOCK_BYTES);
          const uint64_t b_hi = make_smem_desc_sw128(sa + 2 * BLOCK_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t adv = (uint64_t)(k * 32 >> 4);
            const uint32_t first = (kb | k) ? 1u : 0u;
            // B_hi and B_lo tiles are adjacent: A_hi x [B_hi ; B_lo] is one N=256 instruction
            // (hi.hi -> columns [0,128), hi.lo -> [128,256)); lo.hi then accumulates into the latter
            umma_ss<false>(tmem_d, a_hi + adv, b_hi + adv, idesc_cat, first);
            umma_ss<false>(tmem_s, a_lo + adv, b_hi + adv, idesc, 1u);
          }
          tcgen05_commit(&empty[stage]);
          if (kb == nkb - 1) tcgen05_commit(&tfull[acc]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ---- epilogue warps 2..9.  Warps w and w+4 share a TMEM lane quarter and each take half of
    // the tile's 128 columns, 16 at a time: thread = row, all arithmetic in registers, result rows
    // packed into a dense [32][16] box in shared memory and written by TMA.
    const int q = warp & 3;
    const int ew = warp - 2;
    const int half = ew >> 2;                           // which 64 columns of the tile
    unsigned char* stg = staging + ew * STG_BYTES;
    if (lane == 0) { prefetch_tensormap(&tmO_hi); prefetch_tensormap(&tmO_lo); prefetch_tensormap(&tmO_f32); }
    int tc = 0, sidx = 0;
    for (int strip = blockIdx.x; strip < nstrips; strip += gridDim.x, ++sidx) {
      const int wrow0 = strip * BM + q * 32;            // first global row of this warp
      const int grow = wrow0 + lane;                    // this thread's row
      const bool row_ok = grow < p.rows;
      float am = 0.f, ar = 0.f;                         // folded-LN scalars of this row
      if (p.a_sum && row_ok) row_layernorm_scalars(p, grow, am, ar);
      float rsum2[2] = {0.f, 0.f}, rsq2[2] = {0.f, 0.f};   // row sums of the even / odd columns (as the packed fused epilogue)
      // residual of one unit = this row's 16 values of each half of the pair; requested one unit
      // ahead so that its HBM latency overlaps the arithmetic of the current unit
      auto unit_col = [&](int ct_, int un_) {
        int c = ct_ + ct_rot; if (c >= ntile) c -= ntile;
        return c * BN + half * 64 + un_ * UNIT;
      };
      auto load_res = [&](int gc, uint4 (&h)[2], uint4 (&l)[2]) {
        h[0] = h[1] = l[0] = l[1] = make_uint4(0u, 0u, 0u, 0u);
        if (p.res_hi && row_ok && gc < p.N) {
          const size_t o = (size_t)grow * p.N + gc;
          h[0] = __ldg(reinterpret_cast<const uint4*>(p.res_hi + o));
          l[0] = __ldg(reinterpret_cast<const uint4*>(p.res_lo + o));
          if (gc + 8 < p.N) {
            h[1] = __ldg(reinterpret_cast<const uint4*>(p.res_hi + o + 8));
            l[1] = __ldg(reinterpret_cast<const uint4*>(p.res_lo + o + 8));
          }
        }
      };
      uint4 nh[2], nl[2];
      load_res(unit_col(0, 0), nh, nl);
      for (int ct = 0; ct < ntile; ++ct, ++tc) {
        const int acc = tc & 1;
        mbar_wait(&tfull[acc], (tc >> 1) & 1);
        tcgen05_fence_after();
#pragma unroll 1
        for (int un = 0; un < 64 / UNIT; ++un) {
          const int col0 = half * 64 + un * UNIT;       // first column of this unit inside the tile
          const int gc0 = unit_col(ct, un);             // ... and in the output (warp-uniform)
          uint4 rh[2] = {nh[0], nh[1]}, rl[2] = {nl[0], nl[1]};
          {
            int nct = ct, nun = un + 1;
            if (nun == 64 / UNIT) { nun = 0; ++nct; }
            if (nct < ntile) load_res(unit_col(nct, nun), nh, nl);
          }
          if (gc0 >= p.N) continue;
          uint32_t r[UNIT], rs[UNIT];
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 2 * BN + col0;
          tmem_ld_32x16(taddr, r);
          tmem_ld_32x16(taddr + BN, rs);
          tmem_ld_wait();
          float v[UNIT];
#pragma unroll
          for (int j = 0; j < UNIT; j += 4) {
            const bool cok = gc0 + j < p.N;             // N % 4 == 0
            const float4 b4 = *reinterpret_cast<const float4*>(sbias + gc0 + j);
            const float4 s4 = *reinterpret_cast<const float4*>(ss1 + gc0 + j);
            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
            const float ss[4] = {s4.x, s4.y, s4.z, s4.w};
            const __half* h8 = reinterpret_cast<const __half*>(&rh[j >> 3]) + (j & 7);
            const __half* l8 = reinterpret_cast<const __half*>(&rl[j >> 3]) + (j & 7);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float x = __fmaf_rn(__uint_as_float(rs[j + e]), F16_LO_INV, __uint_as_float(r[j + e]));
              if (p.a_sum) x = __fmaf_rn(ar, __fmaf_rn(-am, ss[e], x), bb[e]);    // rho*(acc - mu*s1) + c0
              else x = __fadd_rn(x, bb[e]);
              if (p.res_hi) x = __fadd_rn(x, join_f16(h8[e], l8[e]));
              if (p.relu) x = fmaxf(x, 0.f);
              if (!cok) x = 0.f;
              v[j + e] = x;
              rsum2[e & 1] += x;
              rsq2[e & 1] = __fmaf_rn(x, x, rsq2[e & 1]);
            }
          }
          // the previous TMA store of this warp must have finished reading the staging box
          if (lane == 0) tma_store_wait_read<0>();
          __syncwarp();
          if (p.out_f32) {
            float4* dst = reinterpret_cast<float4*>(stg + lane * (UNIT * 4));
#pragma unroll
            for (int j = 0; j < UNIT; j += 4) dst[j >> 2] = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
            __half hh[UNIT], ll[UNIT];
#pragma unroll
            for (int j = 0; j < UNIT; ++j) split_f16(v[j], hh[j], ll[j]);
            uint4* dh = reinterpret_cast<uint4*>(stg + lane * (UNIT * 2));
            uint4* dl = reinterpret_cast<uint4*>(stg + 32 * UNIT * 2 + lane * (UNIT * 2));
            dh[0] = *reinterpret_cast<uint4*>(&hh[0]); dh[1] = *reinterpret_cast<uint4*>(&hh[8]);
            dl[0] = *reinterpret_cast<uint4*>(&ll[0]); dl[1] = *reinterpret_cast<uint4*>(&ll[8]);
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            if (p.out_f32) {
              tma_store_2d(&tmO_f32, stg, gc0, wrow0);
            } else {
              tma_store_2d(&tmO_hi, stg, gc0, wrow0);
              tma_store_2d(&tmO_lo, stg + 32 * UNIT * 2, gc0, wrow0);
            }
            tma_store_commit();
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
      }
      if (p.out_sum) {
        // row sums of what this strip stored: combine the two column halves of each row
        float* sc = stats + (sidx & 1) * (4 * 32 * 2 * 2);
        float* e = sc + ((q * 32 + lane) * 2 + half) * 2;
        e[0] = rsum2[0] + rsum2[1]; e[1] = rsq2[0] + rsq2[1];
        if (!(e[1] < F16_RANGE_SQ)) atomicOr(&g_refiner_status, 1u);   // range guard (sslam_refiner_range_check)
        named_bar_sync(1, 32 * EPI_WARPS);
        if (half == 0 && row_ok) {
          const float* f = sc + (q * 32 + lane) * 4;
          p.out_sum[grow] = f[0] + f[2];
          p.out_sq[grow] = f[1] + f[3];
        }
      }
    }
    if (lane == 0) tma_store_wait_all<0>();             // all output boxes are in global memory
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2), weight-stationary.  Used whenever K <= 384.
//
// The single-CTA kernel above streams both operands of every 128x128 tile through L2 and shared
// memory (2 x 196 KB per tile at K = 384): at one CTA per SM that saturates the L2 slices and the
// 128 B/cycle shared-memory port long before the tensor pipe.  Here two CTAs on the SMs of one TPC
// share each MMA (M = 256: each CTA owns a 128-row strip and its accumulators; each holds HALF of the
// weight tile), and a pair keeps its 128 weight columns resident for the whole launch:
//   * grid = groups x ceil(N/128) pairs; pair (g, ct) keeps W[ct*128 .. +128, :] (64 rows per CTA,
//     hi+lo, K/64 x 16 KB <= 96 KB) in shared memory and walks the 256-row strip pairs g, g+groups, ...
//   * only activations stream: 32 KB per k-block and CTA, 3 stages; per tile a CTA pulls 196 KB
//     instead of 393 KB through L2 and its MMAs read 6 KB instead of 8 KB of operands each;
//   * the three pairs that own the column tiles of the same strips run in step, so a strip is
//     fetched from DRAM once and served from L2 to the other two;
//   * row statistics for the next folded LayerNorm are written as one partial (sum, sum of squares)
//     per column tile and added up in a fixed order by the consumer (no atomics: results do not
//     depend on scheduling).
// Barriers: TMA of both CTAs signals the LEADER's `full` barriers (rank 0 issues every MMA);
// tcgen05.commit multicasts `empty` / `tfull` to both CTAs; both epilogues arrive on the leader's
// `tempty`.
constexpr int P_STAGES = 3;
constexpr int P_MAX_KB = 6;                               // K <= 384
constexpr int B_HALF = 64 * 128;                          // 64 weight rows x 128 bytes of K
constexpr int P_STAGE_BYTES = 2 * BLOCK_BYTES;            // A_hi, A_lo
constexpr int P_SMEM_B = P_MAX_KB * 2 * B_HALF;
constexpr int P_SMEM_A = P_STAGES * P_STAGE_BYTES;
constexpr int P_SMEM_VECS = 2 * BN * 4;
constexpr int P_SMEM_BARS = (2 * P_STAGES + 5) * 8 + 16;
constexpr int P_SMEM_TOTAL = P_SMEM_B + P_SMEM_A + SMEM_TRANSP + SMEM_STATS + P_SMEM_VECS + P_SMEM_BARS + 1024;

template <bool LN, bool RES, bool RELU, bool OUTF32, bool STATS>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                 const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                 const __grid_constant__ CUtensorMap tmO_hi, const __grid_constant__ CUtensorMap tmO_lo,
                 const __grid_constant__ CUtensorMap tmO_f32, GemmParams p, int groups) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* bres = smem;
  unsigned char* a_stages = smem + P_SMEM_B;
  unsigned char* staging = a_stages + P_SMEM_A;
  float* stats = reinterpret_cast<float*>(staging + SMEM_TRANSP);
  float* sbias = reinterpret_cast<float*>(staging + SMEM_TRANSP + SMEM_STATS);
  float* ss1 = sbias + BN;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + SMEM_TRANSP + SMEM_STATS + P_SMEM_VECS);
  uint64_t* full = bars;
  uint64_t* empty = bars + P_STAGES;
  uint64_t* bfull = bars + 2 * P_STAGES;
  uint64_t* tfull = bfull + 1;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // cluster = the ntile CTA pairs that own the column tiles of the same strips; cluster rank = 2*ct + rank
  const uint32_t crank = cluster_ctarank();
  const uint32_t rank = crank & 1u;                       // rank inside the CTA pair; 0 = MMA leader
  const uint32_t leader = crank & ~1u;                    // cluster rank of this pair's leader
  const int ntile = (p.N + BN - 1) / BN;                  // = multicast width
  const int ct = (int)(crank >> 1), g = blockIdx.x / (2 * ntile);
  const int col_base = ct * BN;
  const int nsp = (p.rows + 2 * BM - 1) / (2 * BM);      // 256-row strip pairs
  const int nkb = (p.K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    // a stage is free again when the MMAs of ALL pairs of the cluster have read it (it is refilled
    // by a multicast that writes every CTA of the same rank)
    // `full` (used in the pair leader): the leader's expect_tx arrival plus one arrival of the peer's
    // producer.  The peer's arrival carries no bytes; it is there so that EVERY producer of the
    // cluster takes part in every use of every stage.  A producer that only waits on `empty` when it
    // is not its turn to fetch could otherwise be overtaken by two phases of that barrier, see the
    // old phase as incomplete again (parity aliasing) and never issue its own stage's loads:
    // a rare deadlock (about one launch in 300 when the epilogue is the bottleneck).
    for (int s = 0; s < P_STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], (uint32_t)ntile); }
    mbar_init(bfull, 1);
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, TMEM_COLS);
  for (int i = threadIdx.x; i < BN; i += NUM_THREADS) {          // this pair's 128 columns of the per-column vectors
    const int c = col_base + i;
    sbias[i] = c < p.N ? __ldg(p.bias + c) : 0.f;
    ss1[i] = (LN && c < p.N) ? __ldg(p.s1 + c) : 0.f;
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {                                            // ---- TMA producer (both CTAs)
      prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmA_lo);
      prefetch_tensormap(&tmB_hi); prefetch_tensormap(&tmB_lo);
      // resident weights: this CTA's 64 of the pair's 128 rows
      const uint32_t bfull_leader = mapa_u32(smem_u32(bfull), leader);
      if (rank == 0) mbar_arrive_expect_tx(bfull, 2u * (uint32_t)nkb * 2u * B_HALF);
      for (int kb = 0; kb < nkb; ++kb) {
        tma_load_2d_pair(bres + kb * 2 * B_HALF, &tmB_hi, bfull_leader, kb * BK, col_base + (int)rank * 64);
        tma_load_2d_pair(bres + kb * 2 * B_HALF + B_HALF, &tmB_lo, bfull_leader, kb * BK, col_base + (int)rank * 64);
      }
      // activations: the ntile CTAs of the same rank need the same 128-row tile of every k-block;
      // they take turns fetching it and multicast it to all of them (L2 -> SM traffic / ntile)
      uint16_t mc_mask = 0;
      for (int j = 0; j < ntile; ++j) mc_mask |= (uint16_t)(1u << (2 * j + (int)rank));
      int stage = 0; uint32_t phase = 0;
      int turn = 0;                                               // running k-block count modulo ntile
      for (int sp = g; sp < nsp; sp += groups) {
        const int row0 = sp * 2 * BM + (int)rank * BM;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          unsigned char* st = a_stages + stage * P_STAGE_BYTES;
          const uint32_t full_leader = mapa_u32(smem_u32(&full[stage]), leader);
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2u * P_STAGE_BYTES);
          else mbar_arrive_cluster(full_leader);
          if (turn == ct) {
            if (ntile == 1) {
              tma_load_2d_pair(st, &tmA_hi, full_leader, kb * BK, row0);
              tma_load_2d_pair(st + BLOCK_BYTES, &tmA_lo, full_leader, kb * BK, row0);
            } else {
              tma_load_2d_pair_mc(st, &tmA_hi, full_leader, kb * BK, row0, mc_mask);
              tma_load_2d_pair_mc(st + BLOCK_BYTES, &tmA_lo, full_leader, kb * BK, row0, mc_mask);
            }
            // the activations come from DRAM (a layer's input is far larger than L2): start the
            // fetch of the same k-block of the NEXT strip pair now, one whole tile ahead
            if (sp + groups < nsp) {
              tma_prefetch_l2_2d(&tmA_hi, kb * BK, row0 + groups * 2 * BM);
              tma_prefetch_l2_2d(&tmA_lo, kb * BK, row0 + groups * 2 * BM);
            }
          }
          if (++turn == ntile) turn = 0;
          if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
        }
      }
      // Producer tail: the last `empty` arrivals of every stage are tcgen05.commit multicasts from
      // the MMA threads of ALL pairs of the cluster, delivered asynchronously into this CTA's shared
      // memory.  Nobody would otherwise wait for them, and the cluster barrier at the end does not
      // order them: if this CTA exited first they would land in the shared memory of whatever CTA
      // runs here next (observed as sporadic launch failures of back-to-back GEMMs).  Drain them.
      for (int i = 0; i < P_STAGES; ++i) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {                               // ---- MMA issuer (leader CTA only)
      const uint32_t idesc = make_instr_desc(FMT_F16, 2 * BM, BN);
      const uint16_t pair_mask = (uint16_t)(3u << leader);        // both CTAs of this pair
      const uint16_t all_mask = (uint16_t)((1u << (2 * ntile)) - 1u);
      int stage = 0; uint32_t phase = 0;
      mbar_wait(bfull, 0);
      tcgen05_fence_after();
      int tc = 0;
      for (int sp = g; sp < nsp; sp += groups, ++tc) {
        const int acc = tc & 1;
        mbar_wait(&tempty[acc], (((uint32_t)tc >> 1) & 1u) ^ 1u);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * 2 * BN;
        const uint32_t tmem_s = tmem_d + BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full[stage], phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(a_stages + stage * P_STAGE_BYTES);
          const uint32_t sb = smem_u32(bres + kb * 2 * B_HALF);
          const uint64_t a_hi = make_smem_desc_sw128(sa);
          const uint64_t a_lo = make_smem_desc_sw128(sa + BLOCK_BYTES);
          const uint64_t b_hi = make_smem_desc_sw128(sb);
          const uint64_t b_lo = make_smem_desc_sw128(sb + B_HALF);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t adv = (uint64_t)(k * 32 >> 4);
            const uint32_t first = (kb | k) ? 1u : 0u;
            umma_ss_pair(tmem_s, a_lo + adv, b_hi + adv, idesc, first);
            umma_ss_pair(tmem_s, a_hi + adv, b_lo + adv, idesc, 1u);
            umma_ss_pair(tmem_d, a_hi + adv, b_hi + adv, idesc, first);
          }
          tcgen05_commit_pair(&empty[stage], all_mask);            // every CTA of the cluster: this pair is done with the stage
          if (kb == nkb - 1) tcgen05_commit_pair(&tfull[acc], pair_mask);
          if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ---- epilogue warps 2..9 of both CTAs, each CTA on its own 128 rows.  The layer's options are
    // template parameters: the per-element code has no branches on kernel arguments (the epilogue
    // is instruction-issue bound — 8 warps share 4 schedulers with the two producer warps).
    const int q = warp & 3;
    const int ew = warp - 2;
    const int half = ew >> 2;
    unsigned char* stg = staging + ew * STG_BYTES;
    if (lane == 0) { prefetch_tensormap(&tmO_hi); prefetch_tensormap(&tmO_lo); prefetch_tensormap(&tmO_f32); }
    const uint32_t tempty_leader0 = mapa_u32(smem_u32(&tempty[0]), leader);
    const uint32_t tempty_leader1 = mapa_u32(smem_u32(&tempty[1]), leader);
    const bool full_cols = col_base + BN <= p.N;          // no ragged columns in this pair's tile
    int tc = 0;
    for (int sp = g; sp < nsp; sp += groups, ++tc) {
      const int wrow0 = sp * 2 * BM + (int)rank * BM + q * 32;
      const int grow = wrow0 + lane;
      const bool row_ok = grow < p.rows;
      float am = 0.f, ar = 0.f, nam = 0.f;
      if (LN && row_ok) { row_layernorm_scalars(p, grow, am, ar); nam = -am; }
      float rsum2[2] = {0.f, 0.f}, rsq2[2] = {0.f, 0.f};   // row sums of the even / odd columns (as the packed fused epilogue)
      // residual of one unit = this row's 16 values of each half of the pair, requested one unit ahead
      const __half* res_h = RES ? p.res_hi + (size_t)(row_ok ? grow : 0) * p.N : nullptr;
      const __half* res_l = RES ? p.res_lo + (size_t)(row_ok ? grow : 0) * p.N : nullptr;
      auto load_res = [&](int gc, uint4 (&h)[2], uint4 (&l)[2]) {
        if (gc + UNIT <= p.N && (p.N & 15) == 0) {      // one 32-byte sector per array: 256-bit loads
          ldg_256(res_h + gc, h);                       // (rows are 32-byte aligned only when N % 16 == 0)
          ldg_256(res_l + gc, l);
        } else {
          h[0] = h[1] = l[0] = l[1] = make_uint4(0u, 0u, 0u, 0u);
          if (gc < p.N) {
            h[0] = __ldg(reinterpret_cast<const uint4*>(res_h + gc));
            l[0] = __ldg(reinterpret_cast<const uint4*>(res_l + gc));
          }
          if (gc + 8 < p.N) {
            h[1] = __ldg(reinterpret_cast<const uint4*>(res_h + gc + 8));
            l[1] = __ldg(reinterpret_cast<const uint4*>(res_l + gc + 8));
          }
        }
      };
      uint4 nh[2], nl[2];
      if (RES) load_res(col_base + half * 64, nh, nl); // in flight while the accumulator completes
      {
        // pull what the NEXT strip pair of this warp will read row-wise (residual pair, LayerNorm
        // partial sums) into L2 now, so that those loads are L2 hits when their turn comes
        const int nrow = grow + groups * 2 * BM;
        if (nrow < p.rows) {
          if (RES) {
            const size_t o = (size_t)nrow * p.N + col_base + half * 64;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p.res_hi + o));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p.res_lo + o));
          }
          if (LN && half == 0 && (lane & 7) == 0) {
            for (int i = 0; i < p.a_parts; ++i) {
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.a_sum + (size_t)i * p.stat_stride + nrow));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.a_sq + (size_t)i * p.stat_stride + nrow));
            }
          }
        }
      }
      const int acc = tc & 1;
      mbar_wait(&tfull[acc], ((uint32_t)tc >> 1) & 1u);
      tcgen05_fence_after();
      uint32_t r[UNIT], rs[UNIT];
      {
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 2 * BN + half * 64;
        tmem_ld_32x16(taddr, r);
        tmem_ld_32x16(taddr + BN, rs);
      }
#pragma unroll
      for (int un = 0; un < 64 / UNIT; ++un) {
        const int col0 = half * 64 + un * UNIT;         // first column of this unit inside the tile
        const int gc0 = col_base + col0;                // ... and in the output (warp-uniform)
        // (one unit ahead only: a deeper prefetch makes ptxas spill, and registers that are the
        // target of an in-flight tcgen05.ld should not be spilled before tcgen05.wait::ld; the
        // Makefile builds with --warn-on-spills.  Requesting the whole slab up front and giving up
        // the accumulator pipelining instead measured 5 % slower.)
        uint4 rh[2], rl[2];
        if (RES) {
          rh[0] = nh[0]; rh[1] = nh[1]; rl[0] = nl[0]; rl[1] = nl[1];
          if (un + 1 < 64 / UNIT) load_res(gc0 + UNIT, nh, nl);
        }
        float v[UNIT];
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < UNIT; ++j) {
          v[j] = __fmaf_rn(__uint_as_float(rs[j]), F16_LO_INV, __uint_as_float(r[j]));   // fold the cross terms
        }
        if (un + 1 < 64 / UNIT) {                       // next unit's accumulators: in flight during the math
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 2 * BN + col0 + UNIT;
          tmem_ld_32x16(taddr, r);
          tmem_ld_32x16(taddr + BN, rs);
        }
        if (gc0 >= p.N) continue;
#pragma unroll
        for (int j = 0; j < UNIT; j += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(sbias + col0 + j);
          const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
          float ss[4] = {0.f, 0.f, 0.f, 0.f};
          if (LN) {
            const float4 s4 = *reinterpret_cast<const float4*>(ss1 + col0 + j);
            ss[0] = s4.x; ss[1] = s4.y; ss[2] = s4.z; ss[3] = s4.w;
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float x = v[j + e];
            if (LN) x = __fmaf_rn(ar, __fmaf_rn(nam, ss[e], x), bb[e]);         // rho*(acc - mu*s1) + c0
            else x = __fadd_rn(x, bb[e]);
            if (RES)
              x = __fadd_rn(__fmaf_rn(__half2float(reinterpret_cast<const __half*>(rl)[j + e]), F16_LO_INV, x),
                            __half2float(reinterpret_cast<const __half*>(rh)[j + e]));
            if (RELU) x = fmaxf(x, 0.f);
            v[j + e] = x;
          }
        }
        if (!full_cols) {                               // ragged last column tile (warp-uniform)
#pragma unroll
          for (int j = 0; j < UNIT; ++j)
            if (gc0 + j >= p.N) v[j] = 0.f;
        }
        if (STATS) {
#pragma unroll
          for (int j = 0; j < UNIT; ++j) { rsum2[j & 1] += v[j]; rsq2[j & 1] = __fmaf_rn(v[j], v[j], rsq2[j & 1]); }
        }
        if (lane == 0) tma_store_wait_read<0>();        // previous box of this warp has left smem
        __syncwarp();
        if (OUTF32) {
          float4* dst = reinterpret_cast<float4*>(stg + lane * (UNIT * 4));
#pragma unroll
          for (int j = 0; j < UNIT; j += 4) dst[j >> 2] = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        } else {
          __half2 hh[UNIT / 2], ll[UNIT / 2];
#pragma unroll
          for (int j = 0; j < UNIT; j += 2) {
            const __half2 h2 = __floats2half2_rn(v[j], v[j + 1]);
            const float2 hf = __half22float2(h2);
            hh[j >> 1] = h2;
            ll[j >> 1] = __floats2half2_rn(__fmul_rn(__fsub_rn(v[j], hf.x), F16_LO_SCALE),
                                           __fmul_rn(__fsub_rn(v[j + 1], hf.y), F16_LO_SCALE));
          }
          uint4* dh = reinterpret_cast<uint4*>(stg + lane * (UNIT * 2));
          uint4* dl = reinterpret_cast<uint4*>(stg + 32 * UNIT * 2 + lane * (UNIT * 2));
          dh[0] = *reinterpret_cast<uint4*>(&hh[0]); dh[1] = *reinterpret_cast<uint4*>(&hh[4]);
          dl[0] = *reinterpret_cast<uint4*>(&ll[0]); dl[1] = *reinterpret_cast<uint4*>(&ll[4]);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (OUTF32) {
            tma_store_2d(&tmO_f32, stg, gc0, wrow0);
          } else {
            tma_store_2d(&tmO_hi, stg, gc0, wrow0);
            tma_store_2d(&tmO_lo, stg + 32 * UNIT * 2, gc0, wrow0);
          }
          tma_store_commit();
        }
      }
      tmem_ld_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(acc ? tempty_leader1 : tempty_leader0);
      if (STATS) {
        // partial row sums of this column tile: combine the two 64-column halves of each row
        float* sc = stats + (tc & 1) * (4 * 32 * 2 * 2);
        float* e = sc + ((q * 32 + lane) * 2 + half) * 2;
        e[0] = rsum2[0] + rsum2[1]; e[1] = rsq2[0] + rsq2[1];
        if (!(e[1] < F16_RANGE_SQ)) atomicOr(&g_refiner_status, 1u);   // range guard (sslam_refiner_range_check)
        named_bar_sync(1, 32 * EPI_WARPS);
        if (half == 0 && row_ok) {
          const float* f = sc + (q * 32 + lane) * 4;
          p.out_sum[(size_t)ct * p.stat_stride + grow] = f[0] + f[2];
          p.out_sq[(size_t)ct * p.stat_stride + grow] = f[1] + f[3];
        }
      }
    }
    if (lane == 0) tma_store_wait_all<0>();
  }
  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// Layer-fused forward: ONE persistent launch runs input projection -> [fc1, fc2 + identity] x blocks
// -> output projection for every row; the activations between layers never reach HBM.
//
// The per-layer kernel above round-trips a [rows, hidden] fp16 pair through HBM for every layer
// (ncu: 12.8 GB per 300 c2 frames against 2.2 GB of input + output), which holds the tensor pipe at
// 40-75 %.  A 128-row strip's activation pair (192 KB) plus the next layer's does not fit in one SM's
// shared memory or TMEM, so the exchange medium is the 126 MB L2 instead:
//   * same cluster shape and data path as gemm_pair_kernel: `ntile` CTA pairs (cta_group::2, M = 256),
//     pair ct owns output columns [128 ct, 128 ct + 128) of EVERY layer; activation k-blocks are TMA-
//     multicast to the pairs; the epilogue threads store their rows of the fp16 pair straight from
//     registers into the scratch, whose layout is the core-matrix operand layout (see SCR_CHUNK below).
//   * a cluster works on chunks of S strip pairs (S x 256 rows).  Order inside a chunk: layer-major,
//     strip-minor (l0: s0..sS-1, l1: s0..sS-1, ...).  The layer outputs go to a per-cluster scratch
//     (h and u pairs, S x 256 rows each: groups x S x 768 KB = ~50 MB for 22 clusters and S = 3) that
//     is rewritten every chunk and therefore stays dirty in L2: after the input rows have been read
//     once, nothing but the final descriptors is written back to DRAM.  fc2 + identity updates h in
//     place (the thread that adds the residual element is the one that stores it).
//   * strip s of layer l+1 may be loaded once all 2*ntile CTAs have stored their columns of strip s of
//     layer l: a publisher warp waits for the CTA's eight epilogue warps, issues ONE release fence at
//     cluster scope and arrives on the `ready[s]` mbarrier of every CTA of the cluster; the producers
//     wait on it and order their TMA loads behind it (fence.proxy.async).  With S >= 3 the wait has
//     more than a tile of slack and never stalls the tensor pipe.
//   * weights are layer-stationary instead of launch-stationary: a dedicated warp reloads the pair's
//     128 weight columns k-block by k-block behind the last strip of the previous layer (`wfree[kb]`
//     is committed by that strip's MMAs, `wfull[kb]` gates the first strip of the next layer), so the
//     switch costs no bubble; 96 KB per CTA and layer out of L2, amortised over S strips.
//   * arithmetic, k order and epilogue are those of gemm_pair_kernel: results are bit-identical to the
//     per-layer path (tests/test_gpu_tc.py).
// Row statistics for the folded LayerNorms and the residual are read back with ld.global.cg: the
// buffers are rewritten inside this launch, so the non-coherent path (ld.global.nc / L1) must not be used.
constexpr int F_MAX_LAYERS = 8;                           // 2 + 2 * blocks, blocks <= 3
constexpr int F_MAX_SLOTS = 4;                            // strip pairs per chunk (S)
constexpr int F_THREADS = NUM_THREADS + 64;               // + the weight producer warp and the publisher warp
constexpr int F_W_WARP = NUM_THREADS / 32;
constexpr int F_PUB_WARP = F_W_WARP + 1;
// Activation stages: F_BK K-elements of the CTA's 128 rows, hi and lo (32 KB).  What bounds the kernel is
// measured in DESIGN.md 4.5: neither the ring depth nor the request size.
constexpr int F_BK = 64;
// Scratch activations (h, u): per 128-row strip and 64-column block one 32 KB piece = exactly one stage of
// the A operand, [hi | lo][column / 8 (8 chunks)][row / 8][row % 8][column % 8] — the no-swizzle core-matrix
// layout of the UMMA descriptor.  A stage is ONE contiguous multicast request; a thread's 8 columns of a chunk
// are 16 contiguous bytes and the 32 rows of a warp 512 contiguous bytes.
constexpr int SCR_CHUNK = (BM / 8) * 64;                   // elements per 8-column chunk (16 core matrices)
constexpr int SCR_PART = 8 * SCR_CHUNK;                    // elements of the hi (or lo) part of a 64-column block
constexpr int SCR_BLOCK = 2 * SCR_PART;                    // elements of a 64-column block of a strip (32 KB)
__device__ __forceinline__ size_t scr_off(int gc) {        // element offset of column gc (a multiple of 8) inside a strip's hi part
  return (size_t)(gc >> 6) * SCR_BLOCK + (size_t)((gc >> 3) & 7) * SCR_CHUNK;
}
constexpr int F_HALF_BYTES = BM * F_BK * 2;               // one 128-row operand tile of a stage
constexpr int F_STAGE_BYTES = 2 * F_HALF_BYTES;           // A_hi, A_lo
// (7 stages of 32 columns, 8 KB per request: 3.4 ms instead of 2.9 — the cost of a multicast request is about
// 160 cycles + 1 cycle per 73 bytes, so the feed wants few, large requests)
static_assert(F_BK == 64, "the stage of the fused kernel is one 64-column block");
// (a fourth 32 KB stage, tried at K = 320 where it fits: 2.60 instead of 2.62 ms — the ring depth is not the limit)
constexpr int F_STAGES = 3;
constexpr int F_SUB = BK / F_BK;                          // stages per 64-element weight k-block
constexpr int F_SMEM_A = F_STAGES * F_STAGE_BYTES;
constexpr int F_SMEM_VECS = F_MAX_LAYERS * 2 * BN * 4;    // [layer][bias 128 | s1 128] of the pair's columns
constexpr int F_SMEM_LN = 2 * BM * 2 * 4;                 // [tile parity][row][-mean, rstd] of the tile's A operand
constexpr int F_NBARS = 2 * F_STAGES + 2 * P_MAX_KB + 4 + F_MAX_SLOTS + 4 + 2;
constexpr int F_SMEM_BARS = F_NBARS * 8 + 16;
constexpr int F_SMEM_TOTAL = P_SMEM_B + F_SMEM_A + F_SMEM_VECS + F_SMEM_LN + F_SMEM_BARS + 1024;
static_assert(F_SMEM_TOTAL <= 227 * 1024, "fused refiner kernel exceeds the shared memory of an SM");

struct FusedMaps {
  CUtensorMap a_hi[3], a_lo[3];      // operand loads: 0 = x (true rows), 1 = h, 2 = u (scratch rows)
  CUtensorMap w_hi[F_MAX_LAYERS], w_lo[F_MAX_LAYERS];
};

struct FusedParams {
  int rows, C, Hd, D, L, S, groups, ntile;
  const float* bias[F_MAX_LAYERS];   // bias, or c0 of a LayerNorm-fed layer
  const float* s1[F_MAX_LAYERS];     // null unless LayerNorm-fed
  __half* s_hi[2];                   // scratch pairs [groups*S*256, Hd]: 0 = h (also the residual), 1 = u
  __half* s_lo[2];
  float* raw;                        // [rows, D] output of the last layer
  float* st_sum[2];                  // partial row sums [2 * ntile][stat_stride]: 0 = of h, 1 = of u
  float* st_sq[2];
  size_t stat_stride;                // = groups * S * 256 scratch rows
};

struct LayerInfo {
  int K, N, src, dst, st_in, st_out;
  bool ln, res, relu, f32, stats;
};
__device__ __forceinline__ LayerInfo layer_info(const FusedParams& p, int l) {
  LayerInfo li;
  const bool first = l == 0, last = l == p.L - 1;
  const bool fc1 = !first && !last && (l & 1), fc2 = !first && !last && !(l & 1);
  li.K = first ? p.C : p.Hd;
  li.N = last ? p.D : p.Hd;
  li.src = first ? 0 : (fc2 ? 2 : 1);
  li.dst = fc1 ? 1 : 0;
  li.st_in = fc2 ? 1 : 0;
  li.st_out = fc1 ? 1 : 0;
  li.ln = fc1 || fc2; li.res = fc2; li.relu = !last; li.f32 = last;
  li.stats = first ? (p.L > 2) : (fc1 || (fc2 && l != p.L - 2));
  return li;
}

__device__ __forceinline__ float ld_cg_f32(const float* p) {
  float v;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void ld_cg_256(const void* ptr, uint4 (&d)[2]) {
  asm volatile("ld.global.cg.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(d[0].x), "=r"(d[0].y), "=r"(d[0].z), "=r"(d[0].w), "=r"(d[1].x), "=r"(d[1].y), "=r"(d[1].z),
                 "=r"(d[1].w)
               : "l"(ptr));
}
__device__ __forceinline__ uint4 ld_cg_128(const void* ptr) {
  uint4 d;
  asm volatile("ld.global.cg.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(d.x), "=r"(d.y), "=r"(d.z), "=r"(d.w) : "l"(ptr));
  return d;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

// what one epilogue warp needs for one tile
struct EpiTile {
  uint32_t tmem_base;
  int q, half, lane, ct, col_base;
  int N, K;                          // layer's output width / LayerNorm width
  size_t srow;                       // this thread's scratch row (statistics)
  size_t soff;                       // element offset of (this row, column 0) in a scratch array (core-matrix layout)
  size_t orow;                       // this thread's row in the output array (scratch row, or true row for the last layer)
  bool row_ok;                       // last layer: orow < rows
  const float* sbias;                // this layer's 128 bias / c0 values of the pair's columns (shared memory)
  const float* ss1;
  __half* o_hi;                      // output pair (scratch h or u)
  __half* o_lo;
  float* o_f32;                      // raw output of the last layer
  const __half* res_h;               // residual pair (scratch h)
  const __half* res_l;
  const float2* ln;                  // (-mean, rstd) of the CTA's 128 rows of the A operand (shared memory)
  uint64_t* lnfull;                  // ... complete when this barrier's phase `ln_parity` is
  uint32_t ln_parity;
  float* out_sum;                    // partial row sums of the output, [2 * ntile][stat_stride]
  float* out_sq;
  size_t stat_stride;
  uint64_t* tfull;
  uint32_t tempty_leader;
};

__device__ __forceinline__ void st_global_256(void* ptr, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(a.x), "r"(a.y), "r"(a.z),
               "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}

// Epilogue of one tile for one warp (32 rows x 64 columns, thread = row, 16 columns per unit).
//
// ONE body for every layer type (the kernel runs all of them, and five unrolled template instances were
// 250 KB of code that the warps of an SM kept evicting from the 32 KB instruction cache): the layer's
// options are data, not code —
//   plain bias      = folded LayerNorm with rho = 1, mu = 0:  fma(1, fma(-0, s1, acc), bias) == acc + bias
//   no ReLU         = max(x, -inf)
//   row statistics  = always accumulated (2 instructions per element), stored only when wanted
// and only the residual loads and the output format are (warp-uniform) branches.
// Outputs leave the registers directly: a thread's 16 values of a unit are 32 contiguous, 32-byte
// aligned bytes of its row in each array of the pair (one full sector: what a TMA box of the same shape
// writes too), so there is no shared-memory staging, no proxy fence and no store queue to wait for
// inside the tile.  Row sums are written per 64-column half (the consumer adds the halves of a column
// tile first, then the tiles: the order of gemm_pair_kernel, bit-identical results).
struct EpiFlags { bool ln, res, relu, f32, stats; };

__device__ __forceinline__ void fused_epilogue_tile(const EpiTile& c, const EpiFlags fl, int acc, uint32_t tfull_parity) {
  const int lane = c.lane, q = c.q, half = c.half;
  const float lo_clamp = fl.relu ? 0.f : __int_as_float(0xff800000);
  const bool wide = (c.N & 15) == 0;                     // fp32 output rows are 32-byte aligned only when N % 16 == 0
  // scratch arrays (h, u) are stored as 8-row x 16-byte core matrices, [strip][column / 8][row / 8][row % 8][column % 8]:
  // a thread's 8 columns of a chunk are 16 contiguous bytes and the 32 rows of a warp make 512 contiguous
  // bytes per chunk, so every load / store instruction of the warp moves four whole 128-byte lines
  const __half* res_h = c.res_h + c.soff;
  const __half* res_l = c.res_l + c.soff;
  uint4 nh[2], nl[2];
  nh[0] = nh[1] = nl[0] = nl[1] = make_uint4(0u, 0u, 0u, 0u);
  auto load_res = [&](int gc) {
    const size_t o = scr_off(gc);
    if (gc < c.N) { nh[0] = ld_cg_128(res_h + o); nl[0] = ld_cg_128(res_l + o); }
    if (gc + 8 < c.N) { nh[1] = ld_cg_128(res_h + o + SCR_CHUNK); nl[1] = ld_cg_128(res_l + o + SCR_CHUNK); }
  };
  if (fl.res) load_res(c.col_base + half * 64);          // in flight while the accumulator completes
  mbar_wait(&c.tfull[acc], tfull_parity);
  tcgen05_fence_after();
  // (-mean, rstd) of this row of the A operand, from the publisher / LayerNorm warp (normally complete a
  // tile ago; never read before lnfull — this warp may get here while other CTAs are still storing the
  // statistics of the strip's previous layer)
  float ar = 1.f, nam = -0.f;
  if (fl.ln) {
    mbar_wait(c.lnfull, c.ln_parity);
    const float2 ln = c.ln[q * 32 + lane];
    nam = ln.x; ar = ln.y;
  }
  uint32_t r[UNIT], rs[UNIT];
  const uint32_t tbase = c.tmem_base + ((uint32_t)(q * 32) << 16) + acc * 2 * BN + half * 64;
  tmem_ld_32x16(tbase, r);
  tmem_ld_32x16(tbase + BN, rs);
  // The arithmetic below is the scalar formula of gemm_pair_kernel's epilogue, element for element
  // (same operations, same roundings), issued two elements at a time: FFMA2 / FADD2 / FMUL2 on register
  // pairs, and the fp16 <-> fp32 mixed forms (FHADD, FHFMA) instead of a conversion plus an fp32 operation.
  // The epilogue is issue bound (two warps per scheduler): this halves its instruction count.
  const uint64_t inv2 = pack_f32x2(F16_LO_INV, F16_LO_INV), ar2 = pack_f32x2(ar, ar), nam2 = pack_f32x2(nam, nam);
  const uint64_t msc2 = pack_f32x2(-F16_LO_SCALE, -F16_LO_SCALE);
  uint64_t sum2 = pack_f32x2(0.f, 0.f), sq2 = sum2;      // row sums of the even / odd columns
#pragma unroll
  for (int un = 0; un < 64 / UNIT; ++un) {
    const int col0 = half * 64 + un * UNIT;
    const int gc0 = c.col_base + col0;
    uint4 rh[2] = {nh[0], nh[1]}, rl[2] = {nl[0], nl[1]};
    if (fl.res && un + 1 < 64 / UNIT) load_res(gc0 + UNIT);
    uint64_t x2[UNIT / 2];
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < UNIT / 2; ++j)                     // fold the cross terms
      x2[j] = ffma2(pack_f32x2(__uint_as_float(rs[2 * j]), __uint_as_float(rs[2 * j + 1])), inv2,
                    pack_f32x2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])));
    if (un + 1 < 64 / UNIT) {                              // next unit's accumulators: in flight during the math
      tmem_ld_32x16(tbase + (un + 1) * UNIT, r);
      tmem_ld_32x16(tbase + (un + 1) * UNIT + BN, rs);
    }
    if (gc0 >= c.N) continue;
    float v[UNIT];
#pragma unroll
    for (int j = 0; j < UNIT / 2; j += 2) {
      const float4 b4 = *reinterpret_cast<const float4*>(c.sbias + col0 + 2 * j);
      const float4 s4 = *reinterpret_cast<const float4*>(c.ss1 + col0 + 2 * j);
      // rho*(acc - mu*s1) + c0
      x2[j] = ffma2(ar2, ffma2(nam2, pack_f32x2(s4.x, s4.y), x2[j]), pack_f32x2(b4.x, b4.y));
      x2[j + 1] = ffma2(ar2, ffma2(nam2, pack_f32x2(s4.z, s4.w), x2[j + 1]), pack_f32x2(b4.z, b4.w));
    }
#pragma unroll
    for (int j = 0; j < UNIT / 2; ++j) unpack_f32x2(x2[j], v[2 * j], v[2 * j + 1]);
    if (fl.res) {
      const uint16_t* ph = reinterpret_cast<const uint16_t*>(rh);
      const uint16_t* pl = reinterpret_cast<const uint16_t*>(rl);
#pragma unroll
      for (int j = 0; j < UNIT; ++j) v[j] = fhadd(ph[j], fhfma(pl[j], F16_LO_INV_BITS, v[j]));   // + (hi + lo * 2^-11)
    }
#pragma unroll
    for (int j = 0; j < UNIT; ++j) v[j] = fmaxf(v[j], lo_clamp);
    if (gc0 + UNIT > c.N) {                                // ragged last column tile (warp-uniform)
#pragma unroll
      for (int j = 0; j < UNIT; ++j) if (gc0 + j >= c.N) v[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < UNIT / 2; ++j) {
      x2[j] = pack_f32x2(v[2 * j], v[2 * j + 1]);
      sum2 = fadd2(sum2, x2[j]);
      sq2 = ffma2(x2[j], x2[j], sq2);
    }
    const bool whole = gc0 + UNIT <= c.N;
    if (fl.f32) {
      if (c.row_ok) {
        float* dst = c.o_f32 + c.orow * (size_t)c.N + gc0;
        if (whole && wide) {
          st_global_256(dst, make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])),
                        make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])));
          st_global_256(dst + 8, make_uint4(__float_as_uint(v[8]), __float_as_uint(v[9]), __float_as_uint(v[10]), __float_as_uint(v[11])),
                        make_uint4(__float_as_uint(v[12]), __float_as_uint(v[13]), __float_as_uint(v[14]), __float_as_uint(v[15])));
        } else {
#pragma unroll
          for (int j = 0; j < UNIT; j += 4)                                            // N % 4 == 0
            if (gc0 + j < c.N) *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
    } else {
      uint32_t hh[UNIT / 2], ll[UNIT / 2];
#pragma unroll
      for (int j = 0; j < UNIT / 2; ++j) {
        const __half2 h2 = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
        const uint32_t hu = *reinterpret_cast<const uint32_t*>(&h2);
        hh[j] = hu;
        // (v - hi) * 2^11 as (hi - v) * -2^11: both steps exact
        const uint64_t d2 = fmul2(pack_f32x2(fhadd((uint16_t)(hu & 0xffffu), -v[2 * j]), fhadd((uint16_t)(hu >> 16), -v[2 * j + 1])), msc2);
        float d0, d1;
        unpack_f32x2(d2, d0, d1);
        const __half2 l2 = __floats2half2_rn(d0, d1);
        ll[j] = *reinterpret_cast<const uint32_t*>(&l2);
      }
      const size_t o = c.soff + scr_off(gc0);
      const uint4* ph = reinterpret_cast<const uint4*>(hh);
      const uint4* pl = reinterpret_cast<const uint4*>(ll);
      *reinterpret_cast<uint4*>(c.o_hi + o) = ph[0];                                   // N % 8 == 0
      *reinterpret_cast<uint4*>(c.o_lo + o) = pl[0];
      if (gc0 + 8 < c.N) {
        *reinterpret_cast<uint4*>(c.o_hi + o + SCR_CHUNK) = ph[1];
        *reinterpret_cast<uint4*>(c.o_lo + o + SCR_CHUNK) = pl[1];
      }
    }
  }
  float rsum, rsq;
  {
    float a0, a1, q0, q1;
    unpack_f32x2(sum2, a0, a1);
    unpack_f32x2(sq2, q0, q1);
    rsum = a0 + a1; rsq = q0 + q1;
  }
  // range guard: the pair just stored is garbage once an |x| reaches 65504 (x^2 alone then exceeds the
  // bound; NaN / inf fail the comparison too)
  if (!fl.f32 && !(rsq < F16_RANGE_SQ)) atomicOr(&g_refiner_status, 1u);
  tmem_ld_wait();
  tcgen05_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(c.tempty_leader);
  if (fl.stats) {                                        // partial row sums of this warp's 64 columns
    const size_t o = (size_t)(2 * c.ct + half) * c.stat_stride + c.srow;
    c.out_sum[o] = rsum;
    c.out_sq[o] = rsq;
  }
}

__global__ void __launch_bounds__(F_THREADS, 1)
refiner_fused_kernel(const __grid_constant__ FusedMaps tm, const FusedParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* bres = smem;
  unsigned char* a_stages = smem + P_SMEM_B;
  float* svec = reinterpret_cast<float*>(a_stages + F_SMEM_A);                    // [L][bias 128 | s1 128]
  float2* sln = reinterpret_cast<float2*>(a_stages + F_SMEM_A + F_SMEM_VECS);     // [tile parity][row] (-mean, rstd)
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_stages + F_SMEM_A + F_SMEM_VECS + F_SMEM_LN);
  uint64_t* full = bars;
  uint64_t* empty = full + F_STAGES;
  uint64_t* wfull = empty + F_STAGES;
  uint64_t* wfree = wfull + P_MAX_KB;
  uint64_t* tfull = wfree + P_MAX_KB;
  uint64_t* tempty = tfull + 2;
  uint64_t* ready = tempty + 2;
  uint64_t* tdone = ready + F_MAX_SLOTS;
  uint64_t* lnfull = tdone + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(lnfull + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const uint32_t rank = crank & 1u;
  const uint32_t leader = crank & ~1u;
  const int ntile = p.ntile;
  const int ct = (int)(crank >> 1), g = blockIdx.x / (2 * ntile);
  const int col_base = ct * BN;
  const int groups = p.groups;
  const int nsp = (p.rows + 2 * BM - 1) / (2 * BM);
  const int cnt = (nsp - g + groups - 1) / groups;        // strip pairs of this cluster: g, g + groups, ...
  const int L = p.L, S = p.S;

  if (threadIdx.x == 0) {
    for (int s = 0; s < F_STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], (uint32_t)ntile); }
    for (int k = 0; k < P_MAX_KB; ++k) { mbar_init(&wfull[k], 1); mbar_init(&wfree[k], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * EPI_WARPS); }
    for (int s = 0; s < F_MAX_SLOTS; ++s) mbar_init(&ready[s], (uint32_t)(2 * ntile));
    for (int i = 0; i < 4; ++i) mbar_init(&tdone[i], EPI_WARPS);
    for (int i = 0; i < 2; ++i) mbar_init(&lnfull[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, TMEM_COLS);
  for (int i = threadIdx.x; i < L * BN; i += F_THREADS) {        // this pair's 128 columns of every layer's vectors
    const int l = i / BN, c = col_base + (i - l * BN);
    const int N = (l == L - 1) ? p.D : p.Hd;
    svec[l * 2 * BN + (i - l * BN)] = c < N ? __ldg(p.bias[l] + c) : 0.f;
    svec[l * 2 * BN + BN + (i - l * BN)] = (p.s1[l] && c < N) ? __ldg(p.s1[l] + c) : 0.f;
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---- activation producer (every CTA): one thread drives the barriers and the TMA.  It never does
    // anything else: with three stages in flight any pause of this thread is a bubble in the tensor pipe.
    if (lane == 0) for (int i = 0; i < 3; ++i) { prefetch_tensormap(&tm.a_hi[i]); prefetch_tensormap(&tm.a_lo[i]); }
    uint16_t mc_mask = 0;
    for (int j = 0; j < ntile; ++j) mc_mask |= (uint16_t)(1u << (2 * j + (int)rank));
    const int nkb0 = (p.C + F_BK - 1) / F_BK;
    const int scr_kb = (p.Hd + F_BK - 1) / F_BK;                  // 64-column blocks of a scratch strip
    int stage = 0; uint32_t phase = 0;
    int turn = 0, nchunk = 0;
    for (int c0 = 0; c0 < cnt; c0 += S, ++nchunk) {
      const int Sc = min(S, cnt - c0);
      for (int l = 0; l < L; ++l) {
        const LayerInfo li = layer_info(p, l);
        const int nkb = (li.K + F_BK - 1) / F_BK;            // stages per tile
        const CUtensorMap* mh = &tm.a_hi[li.src];
        const CUtensorMap* ml = &tm.a_lo[li.src];
        for (int s = 0; s < Sc; ++s) {
          const int srow0 = ((g * S + s) * 2 + (int)rank) * BM;
          const int row0 = li.src == 0 ? (g + (c0 + s) * groups) * 2 * BM + (int)rank * BM : srow0;
          if (l > 0) {
            if (lane == 0) {
              // every CTA of the cluster has stored its columns of this strip's previous layer and
              // published them (release fence at cluster scope + arrival).  What follows reads the strip
              // only through L2 (TMA here, ld.global.cg in the other warps), in program order after the
              // wait: no cluster-scope acquire fence, which on this hardware is an invalidation of the
              // whole L1 (CCTL.IVALL) and would evict the bias vectors the epilogue reads through it
              // once per tile.  The proxy fence orders the async proxy (TMA) after the wait.
              const uint32_t par = (uint32_t)(nchunk * (L - 1) + l - 1) & 1u;
              mbar_wait(&ready[s], par);
              fence_proxy_async_all();
            }
          }
          if (lane == 0) {
            const bool pf = (l == L - 1) && (c0 + S + s < cnt);   // next chunk's input rows -> L2
            const int pf_row = (g + (c0 + S + s) * groups) * 2 * BM + (int)rank * BM;
            for (int kb = 0; kb < nkb; ++kb) {
              mbar_wait(&empty[stage], phase ^ 1);
              unsigned char* st = a_stages + stage * F_STAGE_BYTES;
              const uint32_t full_leader = mapa_u32(smem_u32(&full[stage]), leader);
              if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2u * F_STAGE_BYTES);
              else mbar_arrive_cluster(full_leader);
              if (turn == ct) {
                // x: box of the row-major pair (128 rows x 64 columns, 128-byte swizzle); h / u: the stage is
                // 16 KB of contiguous memory (8 chunks of the strip), fetched as 16 rows of 1 KB of a flat map
                const int c0x = li.src == 0 ? kb * F_BK : 0;
                const int c1x = li.src == 0 ? row0 : ((srow0 / BM) * scr_kb + kb) * (F_STAGE_BYTES / 1024);
                if (li.src != 0) {                              // one 32 KB request: hi and lo of the block
                  if (ntile == 1) tma_load_2d_pair(st, mh, full_leader, 0, c1x);
                  else tma_load_2d_pair_mc(st, mh, full_leader, 0, c1x, mc_mask);
                } else if (ntile == 1) {
                  tma_load_2d_pair(st, mh, full_leader, c0x, c1x);
                  tma_load_2d_pair(st + F_HALF_BYTES, ml, full_leader, c0x, c1x);
                } else {
                  tma_load_2d_pair_mc(st, mh, full_leader, c0x, c1x, mc_mask);
                  tma_load_2d_pair_mc(st + F_HALF_BYTES, ml, full_leader, c0x, c1x, mc_mask);
                }
                if (pf && kb < nkb0) {
                  tma_prefetch_l2_2d(&tm.a_hi[0], kb * F_BK, pf_row);
                  tma_prefetch_l2_2d(&tm.a_lo[0], kb * F_BK, pf_row);
                }
              }
              if (++turn == ntile) turn = 0;
              if (++stage == F_STAGES) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
    if (lane == 0) {
      for (int i = 0; i < F_STAGES; ++i) {                        // drain the last multicast commits (see gemm_pair_kernel)
        mbar_wait(&empty[stage], phase ^ 1);
        if (++stage == F_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == F_W_WARP) {
    if (elect_one()) {                                            // ---- weight producer (every CTA)
      const uint32_t wfull_leader0 = mapa_u32(smem_u32(&wfull[0]), leader);
      uint32_t n = 0;                                             // running (chunk, layer) count
      for (int c0 = 0; c0 < cnt; c0 += S) {
        for (int l = 0; l < L; ++l, ++n) {
          const LayerInfo li = layer_info(p, l);
          const int nkb = (li.K + BK - 1) / BK;
          prefetch_tensormap(&tm.w_hi[l]); prefetch_tensormap(&tm.w_lo[l]);
          for (int kb = 0; kb < P_MAX_KB; ++kb) {
            // the last strip of the previous layer has multiplied by this k-block of the old weights
            if (n > 0) mbar_wait(&wfree[kb], (n - 1) & 1u);
            if (kb < nkb) {
              if (rank == 0) mbar_arrive_expect_tx(&wfull[kb], 2u * 2u * B_HALF);
              tma_load_2d_pair(bres + kb * 2 * B_HALF, &tm.w_hi[l], wfull_leader0 + 8u * kb, kb * BK, col_base + (int)rank * 64);
              tma_load_2d_pair(bres + kb * 2 * B_HALF + B_HALF, &tm.w_lo[l], wfull_leader0 + 8u * kb, kb * BK, col_base + (int)rank * 64);
            } else if (rank == 0) {
              mbar_arrive(&wfull[kb]);                            // keeps the phase count of unused k-blocks in step
            }
          }
        }
      }
      // the last layer's wfree commits (multicast into this CTA) must have landed before the CTA may exit
      for (int kb = 0; kb < P_MAX_KB; ++kb) mbar_wait(&wfree[kb], (n - 1) & 1u);
    }
  } else if (warp == F_PUB_WARP) {
    // ---- publisher / LayerNorm warp.  Two jobs, both off the critical paths of the other warps:
    //  P(l, s): when the eight epilogue warps have stored tile (l, s) (tdone), lane 0 issues ONE release
    //           fence at cluster scope (cumulative over their stores) and one arrival per CTA of the
    //           cluster on ready[s]; the fence's round trip to L2 is paid here, not by the epilogue;
    //  N(l, s): once ready[s] of layer l-1 has completed, the warp turns the partial row sums of the
    //           strip into the (-mean, rstd) pairs of this CTA's 128 rows (shared memory) and completes
    //           lnfull[tile parity]; the epilogue threads then need one 8-byte shared load per tile.
    // Order: N of the NEXT tile, then P of the current one (the next tile's scalars are ready a whole
    // tile before its epilogue starts); with single-strip chunks the next tile depends on the current
    // one, so P comes first.  Two (-mean, rstd) buffers, by tile parity: N(t + 1) overwrites what tile
    // t - 1 read, and the P(t - 1) before it has waited for that tile's epilogue.
    const uint32_t ncta = (uint32_t)(2 * ntile);
    uint32_t tcn = 0, t = 0;                                      // published tiles / all tiles so far
    int nchunk = 0;
    auto ln_tile = [&](uint32_t t1, int nch, int l, int s) {      // N for the tile with running index t1
      const LayerInfo li = layer_info(p, l);
      if (l >= 1 && li.ln) {
        if (lane == 0) {
          mbar_wait(&ready[s], (uint32_t)(nch * (L - 1) + l - 1) & 1u);
        }
        __syncwarp();
        const int srow0 = ((g * S + s) * 2 + (int)rank) * BM;
        const float* ps = p.st_sum[li.st_in];
        const float* pq = p.st_sq[li.st_in];
        constexpr int MAXP = 2 * (P_MAX_KB * BK / BN);             // partial sums per row: two halves per column tile
        float vs[BM / 32][MAXP], vq[BM / 32][MAXP];
#pragma unroll
        for (int rr = 0; rr < BM / 32; ++rr)                       // all loads first: one L2 round trip for the lot
#pragma unroll
          for (int i = 0; i < MAXP; ++i) {
            const size_t o = (size_t)i * p.stat_stride + (size_t)(srow0 + rr * 32 + lane);
            vs[rr][i] = i < 2 * ntile ? ld_cg_f32(ps + o) : 0.f;
            vq[rr][i] = i < 2 * ntile ? ld_cg_f32(pq + o) : 0.f;
          }
#pragma unroll
        for (int rr = 0; rr < BM / 32; ++rr) {                     // fixed order: halves of a column tile, then tiles
          float sm = 0.f, sq = 0.f;
#pragma unroll
          for (int i = 0; i < MAXP; i += 2)
            if (i < 2 * ntile) { sm += vs[rr][i] + vs[rr][i + 1]; sq += vq[rr][i] + vq[rr][i + 1]; }
          const float mean = sm / (float)li.K;
          const float var = fmaxf(sq / (float)li.K - mean * mean, 0.f);
          sln[(t1 & 1u) * BM + rr * 32 + lane] = make_float2(-mean, 1.0f / sqrtf(var + 1e-5f));
        }
        __syncwarp();
      }
      if (lane == 0) mbar_arrive(&lnfull[t1 & 1u]);               // one phase per tile, LayerNorm-fed or not
    };
    ln_tile(0, 0, 0, 0);
    for (int c0 = 0; c0 < cnt; c0 += S, ++nchunk) {
      const int Sc = min(S, cnt - c0);
      for (int l = 0; l < L; ++l) {
        for (int s = 0; s < Sc; ++s, ++t) {
          // the tile that follows (l, s) in the cluster's order
          int nch = nchunk, nl = l, ns = s + 1;
          if (ns == Sc) { ns = 0; ++nl; }
          if (nl == L) { nl = 0; ++nch; }
          const bool have_next = nl < L && (nch == nchunk || c0 + S < cnt);
          // it depends on the current tile only when the chunk has a single strip
          const bool next_first = !(Sc == 1 && nch == nchunk);
          if (have_next && next_first) ln_tile(t + 1, nch, nl, ns);
          if (l + 1 < L) {                                        // P(l, s)
            if (lane == 0) {
              mbar_wait(&tdone[tcn & 3u], (tcn >> 2) & 1u);
              asm volatile("fence.release.cluster;" ::: "memory");
              const uint32_t rb = smem_u32(&ready[s]);
              for (uint32_t j = 0; j < ncta; ++j) mbar_arrive_cluster_relaxed(mapa_u32(rb, j));
            }
            ++tcn;
          }
          if (have_next && !next_first) ln_tile(t + 1, nch, nl, ns);
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {                               // ---- MMA issuer (leader CTA of each pair)
      const uint32_t idesc = make_instr_desc(FMT_F16, 2 * BM, BN);
      const uint16_t pair_mask = (uint16_t)(3u << leader);
      const uint16_t all_mask = (uint16_t)((1u << (2 * ntile)) - 1u);
      int stage = 0; uint32_t phase = 0;
      uint32_t tc = 0, n = 0;
      for (int c0 = 0; c0 < cnt; c0 += S) {
        const int Sc = min(S, cnt - c0);
        for (int l = 0; l < L; ++l, ++n) {
          const LayerInfo li = layer_info(p, l);
          const int nkb = (li.K + BK - 1) / BK;               // weight k-blocks of this layer
          for (int s = 0; s < Sc; ++s, ++tc) {
            const int acc = (int)(tc & 1u);
            mbar_wait(&tempty[acc], ((tc >> 1) & 1u) ^ 1u);
            tcgen05_fence_after();
            const uint32_t tmem_d = tmem_base + acc * 2 * BN;
            const uint32_t tmem_s = tmem_d + BN;
            const bool last_strip = s == Sc - 1;
            const int nst = (li.K + F_BK - 1) / F_BK;             // activation stages of this tile (32 K-elements each)
            for (int ks = 0; ks < nst; ++ks) {
              const int kb = ks / F_SUB, sub = ks % F_SUB;        // weight k-block (64 K-elements) of this stage
              if (s == 0 && sub == 0) mbar_wait(&wfull[kb], n & 1u);     // this layer's weights, k-block kb
              mbar_wait(&full[stage], phase);
              tcgen05_fence_after();
              const uint32_t sa = smem_u32(a_stages + stage * F_STAGE_BYTES);
              const uint32_t sb = smem_u32(bres + kb * 2 * B_HALF);
              // x tiles are 128-byte-swizzled rows; h / u tiles are core matrices (no swizzle): next chunk
              // of K at +2048 bytes, next 8 rows at +128 bytes, a k-step (two chunks) every 4096 bytes
              const bool cm = li.src != 0;
              const uint64_t a_hi = cm ? make_smem_desc_interleave(sa, 2048, 128) : make_smem_desc_sw128(sa);
              const uint64_t a_lo = cm ? make_smem_desc_interleave(sa + F_HALF_BYTES, 2048, 128)
                                       : make_smem_desc_sw128(sa + F_HALF_BYTES);
              const uint64_t a_step = cm ? (uint64_t)(4096 >> 4) : (uint64_t)(32 >> 4);
              const uint64_t boff = (uint64_t)(sub * F_BK * 2 >> 4);      // position inside the 128-byte weight rows
              const uint64_t b_hi = make_smem_desc_sw128(sb) + boff;
              const uint64_t b_lo = make_smem_desc_sw128(sb + B_HALF) + boff;
              // a pair whose columns lie beyond the layer's width (output projection narrower than the hidden
              // layers) keeps the barrier protocol going but issues no MMAs: its epilogue skips every column
              if (col_base < li.N)
#pragma unroll
              for (int k = 0; k < F_BK / 16; ++k) {
                const uint64_t adv = (uint64_t)(k * 32 >> 4), aadv = (uint64_t)k * a_step;
                const uint32_t first = (ks | k) ? 1u : 0u;
                umma_ss_pair(tmem_s, a_lo + aadv, b_hi + adv, idesc, first);
                umma_ss_pair(tmem_s, a_hi + aadv, b_lo + adv, idesc, 1u);
                umma_ss_pair(tmem_d, a_hi + aadv, b_hi + adv, idesc, first);
              }
              tcgen05_commit_pair(&empty[stage], all_mask);
              if (last_strip && (sub == F_SUB - 1 || ks == nst - 1)) tcgen05_commit_pair(&wfree[kb], pair_mask);
              if (ks == nst - 1) tcgen05_commit_pair(&tfull[acc], pair_mask);
              if (++stage == F_STAGES) { stage = 0; phase ^= 1; }
            }
            if (last_strip)
              for (int kb = nkb; kb < P_MAX_KB; ++kb) tcgen05_commit_pair(&wfree[kb], pair_mask);
          }
        }
      }
    }
  } else {
    // ---- epilogue warps 2..9 of both CTAs
    EpiTile c;
    c.tmem_base = tmem_base;
    c.q = warp & 3;
    const int ew = warp - 2;
    c.half = ew >> 2;
    c.lane = lane; c.ct = ct; c.col_base = col_base;
    c.o_f32 = p.raw;
    c.res_h = p.s_hi[0]; c.res_l = p.s_lo[0];
    c.stat_stride = p.stat_stride;
    c.tfull = tfull;
    const uint32_t tempty_leader0 = mapa_u32(smem_u32(&tempty[0]), leader);
    const uint32_t tempty_leader1 = mapa_u32(smem_u32(&tempty[1]), leader);
    uint32_t tc = 0;
    uint32_t tcn = 0;                                            // tiles handed to the publisher so far
    int nchunk = 0;
    const size_t scr_strip = (size_t)((p.Hd + F_BK - 1) / F_BK) * SCR_BLOCK;   // elements of one strip of a scratch array
    for (int c0 = 0; c0 < cnt; c0 += S, ++nchunk) {
      for (int l = 0; l < L; ++l) {
        const LayerInfo li = layer_info(p, l);
        c.N = li.N; c.K = li.K;
        c.sbias = svec + l * 2 * BN; c.ss1 = c.sbias + BN;
        c.o_hi = p.s_hi[li.dst]; c.o_lo = p.s_lo[li.dst];
        c.out_sum = p.st_sum[li.st_out]; c.out_sq = p.st_sq[li.st_out];
        // s < min(S, cnt - c0), written so that no chunk count stays live across the tile (168 registers, no spill)
        for (int s = 0; s < S && c0 + s < cnt; ++s, ++tc) {
          const int srow_w = ((g * S + s) * 2 + (int)rank) * BM + c.q * 32;       // scratch row of lane 0
          const int trow_w = (g + (c0 + s) * groups) * 2 * BM + (int)rank * BM + c.q * 32;
          c.srow = (size_t)(srow_w + lane);
          c.soff = (size_t)((g * S + s) * 2 + (int)rank) * scr_strip + (size_t)(((c.q * 32 + lane) >> 3) * 64 + (lane & 7) * 8);
          c.orow = li.f32 ? (size_t)(trow_w + lane) : c.srow;
          c.row_ok = trow_w + lane < p.rows;
          const int acc = (int)(tc & 1u);
          const uint32_t par = (tc >> 1) & 1u;
          c.tempty_leader = acc ? tempty_leader1 : tempty_leader0;
          const EpiFlags fl{li.ln, li.res, li.relu, li.f32, li.stats};
          c.ln = sln + (tc & 1u) * BM;
          c.lnfull = &lnfull[tc & 1u];
          c.ln_parity = (tc >> 1) & 1u;
          fused_epilogue_tile(c, fl, acc, par);
          if (l < L - 1) {                                        // hand the tile to the publisher warp
            __syncwarp();
            if (lane == 0) mbar_arrive(&tdone[tcn & 3u]);
            ++tcn;
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// fp32 [n] -> fp16 pair
__global__ void split_kernel(const float4* __restrict__ src, uint2* __restrict__ hi, uint2* __restrict__ lo,
                             size_t n4) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) {
    const float4 x = __ldg(src + i);
    __half h[4], l[4];
    split_f16(x.x, h[0], l[0]); split_f16(x.y, h[1], l[1]);
    split_f16(x.z, h[2], l[2]); split_f16(x.w, h[3], l[3]);
    hi[i] = *reinterpret_cast<uint2*>(h);
    lo[i] = *reinterpret_cast<uint2*>(l);
  }
}

// Weight folding for a Linear fed by LayerNorm(gamma, beta): one warp per output row n.
//   W'[n,k] = W[n,k] * gamma[k]  -> fp16 pair;  s1[n] = sum_k W'[n,k] (of the pair actually used);
//   c0[n] = sum_k beta[k] * W[n,k] + bias[n]
__global__ void fold_ln_kernel(const float* __restrict__ W, const float* __restrict__ gamma,
                               const float* __restrict__ beta, const float* __restrict__ bias, int N, int K,
                               __half* __restrict__ hi, __half* __restrict__ lo, float* __restrict__ s1,
                               float* __restrict__ c0) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  float a = 0.f, c = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = W[(size_t)n * K + k];
    const float wp = __fmul_rn(w, gamma[k]);
    __half h, l;
    split_f16(wp, h, l);
    hi[(size_t)n * K + k] = h;
    lo[(size_t)n * K + k] = l;
    a += join_f16(h, l);
    c = __fmaf_rn(beta[k], w, c);
  }
  a = warp_reduce_sum(a);
  c = warp_reduce_sum(c);
  if (lane == 0) { s1[n] = a; c0[n] = c + bias[n]; }
}

struct Pair { __half* hi; __half* lo; };

int launch_split(const float* src, Pair dst, size_t n, cudaStream_t stream) {
  SSLAM_LAUNCH(KK_SPLIT, stream,
               split_kernel<<<num_sms() * 8, 256, 0, stream>>>(reinterpret_cast<const float4*>(src),
                                                               reinterpret_cast<uint2*>(dst.hi),
                                                               reinterpret_cast<uint2*>(dst.lo), n / 4));
  return SSLAM_OK;
}

struct RowStats { float* sum; float* sq; int parts; };   // [parts][stat_stride] partial row sums

size_t stat_stride_of(int rows) { return align_up((size_t)rows, 64); }
int stat_parts_of(int N) { return (N + BN - 1) / BN; }

int launch_gemm(Pair a, Pair w, int rows, int N, int K, const float* bias, RowStats a_ln, const float* s1,
                Pair residual, int relu, float* out_f32, Pair out, RowStats* out_stats, cudaStream_t stream) {
  // weight-stationary CTA-pair kernel: weights must fit (K <= 384) and the ntile pairs form one cluster
  const bool pair = (K + BK - 1) / BK <= P_MAX_KB && (N + BN - 1) / BN <= 4;
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo;
  int rc;
  if ((rc = make_tensor_map_2d(&ta_hi, a.hi, rows, K, BM, BK, 2))) return rc;
  if ((rc = make_tensor_map_2d(&ta_lo, a.lo, rows, K, BM, BK, 2))) return rc;
  if ((rc = make_tensor_map_2d(&tb_hi, w.hi, N, K, pair ? 64 : BN, BK, 2))) return rc;
  if ((rc = make_tensor_map_2d(&tb_lo, w.lo, N, K, pair ? 64 : BN, BK, 2))) return rc;
  // outputs: dense [32 rows][16 cols] boxes, no swizzle; unused maps alias a valid one
  CUtensorMap to_hi, to_lo, to_f32;
  if (out.hi) {
    if ((rc = make_tensor_map_2d(&to_hi, out.hi, rows, N, 32, UNIT, 2, 0))) return rc;
    if ((rc = make_tensor_map_2d(&to_lo, out.lo, rows, N, 32, UNIT, 2, 0))) return rc;
    to_f32 = to_hi;
  } else {
    if ((rc = make_tensor_map_2d(&to_f32, out_f32, rows, N, 32, UNIT, 4, 0))) return rc;
    to_hi = to_f32; to_lo = to_f32;
  }
  static DeviceOnce once;
  if (once.first_use()) {
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(gemm_f16x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          SMEM_TOTAL));
  }
  GemmParams gp;
  gp.rows = rows; gp.N = N; gp.K = K; gp.bias = bias; gp.res_hi = residual.hi; gp.res_lo = residual.lo;
  gp.relu = relu; gp.out_f32 = out_f32; gp.out_hi = out.hi; gp.out_lo = out.lo;
  gp.a_sum = a_ln.sum; gp.a_sq = a_ln.sq; gp.a_parts = a_ln.parts; gp.s1 = s1;
  gp.out_sum = out_stats ? out_stats->sum : nullptr;
  gp.out_sq = out_stats ? out_stats->sq : nullptr;
  gp.stat_stride = stat_stride_of(rows);
  if (pair) {
    const int ntile = (N + BN - 1) / BN;
    const int nsp = (rows + 2 * BM - 1) / (2 * BM);
    int groups = 0;
    if (out_stats) out_stats->parts = ntile;
    const bool ln = a_ln.sum != nullptr, res = residual.hi != nullptr, st = out_stats != nullptr;
#define SSLAM_PAIR_LAUNCH(LN_, RES_, RELU_, F32_, ST_)                                                     \
  do {                                                                                                     \
    auto kfn = gemm_pair_kernel<LN_, RES_, RELU_, F32_, ST_>;                                              \
    static std::atomic<int> max_clusters[64][5] = {};             /* per device and cluster shape, 0 = not queried */ \
    int dev_ = 0;                                                                                          \
    SSLAM_CHECK_CUDA(cudaGetDevice(&dev_));                                                                \
    dev_ &= 63;                                                                                            \
    cudaLaunchConfig_t cfg = {};                                                                           \
    cudaLaunchAttribute attr[1];                                                                           \
    attr[0].id = cudaLaunchAttributeClusterDimension;                                                      \
    attr[0].val.clusterDim.x = 2 * ntile; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;      \
    cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = P_SMEM_TOTAL; cfg.stream = stream;            \
    cfg.attrs = attr; cfg.numAttrs = 1;                                                                    \
    int mcl = max_clusters[dev_][ntile].load();                                                               \
    if (mcl == 0) {                                                                                        \
      SSLAM_CHECK_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_TOTAL)); \
      cfg.gridDim = dim3(2 * ntile);                                                                       \
      SSLAM_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&mcl, kfn, &cfg));                                   \
      SSLAM_REQUIRE(mcl >= 1, SSLAM_EUNSUPPORTED, "refiner: no cluster of %d CTAs fits on this device", 2 * ntile); \
      max_clusters[dev_][ntile].store(mcl);                                                                \
    }                                                                                                      \
    groups = mcl < nsp ? mcl : nsp;                               /* all clusters co-resident */            \
    cfg.gridDim = dim3(2u * ntile * groups);                                                               \
    SSLAM_LAUNCH(KK_GEMM, stream,                                                                          \
                 cudaLaunchKernelEx(&cfg, kfn, ta_hi, ta_lo, tb_hi, tb_lo, to_hi, to_lo, to_f32, gp, groups)); \
  } while (0)
    // the layer shapes of DescriptorRefiner: input projection, fc1, fc2 (+identity), output projection
    if (!ln && !res && relu && !out_f32 && st) SSLAM_PAIR_LAUNCH(false, false, true, false, true);
    else if (!ln && !res && relu && !out_f32 && !st) SSLAM_PAIR_LAUNCH(false, false, true, false, false);
    else if (ln && !res && relu && !out_f32 && st) SSLAM_PAIR_LAUNCH(true, false, true, false, true);
    else if (ln && res && relu && !out_f32 && st) SSLAM_PAIR_LAUNCH(true, true, true, false, true);
    else if (ln && res && relu && !out_f32 && !st) SSLAM_PAIR_LAUNCH(true, true, true, false, false);
    else if (!ln && !res && !relu && out_f32 && !st) SSLAM_PAIR_LAUNCH(false, false, false, true, false);
    else SSLAM_REQUIRE(false, SSLAM_EUNSUPPORTED, "refiner: layer option combination not instantiated");
#undef SSLAM_PAIR_LAUNCH
    return SSLAM_OK;
  }
  if (out_stats) out_stats->parts = 1;
  const int strips = (rows + BM - 1) / BM;
  const int grid = strips < num_sms() ? strips : num_sms();        // persistent: one CTA per SM
  SSLAM_LAUNCH(KK_GEMM, stream,
               gemm_f16x3_kernel<<<grid, NUM_THREADS, SMEM_TOTAL, stream>>>(ta_hi, ta_lo, tb_hi, tb_lo, to_hi, to_lo,
                                                                            to_f32, gp));
  return SSLAM_OK;
}

// ---- host side of the fused kernel
bool fused_eligible(int C, int Hd, int D, int blocks) {
  const int nt = (Hd + BN - 1) / BN;
  return g_refiner_fused > 0 && C <= P_MAX_KB * BK && Hd <= P_MAX_KB * BK && D <= nt * BN &&
         2 + 2 * blocks <= F_MAX_LAYERS;
}
// upper bound of the scratch rows: clusters that can be co-resident (<= 160 SMs / cluster size) x S x 256
size_t fused_scratch_rows(int rows, int Hd) {
  const size_t nt = (size_t)(Hd + BN - 1) / BN;
  const size_t nsp = ((size_t)rows + 2 * BM - 1) / (2 * BM);
  const size_t cap = 160 / (2 * nt);
  return (nsp < cap ? nsp : cap) * F_MAX_SLOTS * 2 * BM;
}
size_t fused_scratch_bytes(int rows, int Hd) {
  const size_t r = fused_scratch_rows(rows, Hd), nt = (size_t)(Hd + BN - 1) / BN;
  const size_t hd_pad = (size_t)(Hd + F_BK - 1) / F_BK * F_BK;     // strips hold whole 64-column blocks
  return 2 * 2 * align_up(r * hd_pad * 2, 1024) + 4 * align_up(2 * nt * r * 4, 256) + 2048;
}

struct FusedLayer { Pair w; const float* bias; const float* s1; };

int launch_fused(Pair xs, const FusedLayer* layers, int rows, int C, int Hd, int D, int blocks, float* raw,
                 char* scratch, cudaStream_t stream) {
  const int L = 2 + 2 * blocks;
  const int ntile = (Hd + BN - 1) / BN;
  const int nsp = (rows + 2 * BM - 1) / (2 * BM);
  static std::atomic<int> max_clusters[64][5] = {};              // per device and cluster shape, 0 = not queried
  int dev = 0;
  SSLAM_CHECK_CUDA(cudaGetDevice(&dev));
  dev &= 63;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2 * ntile; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(F_THREADS); cfg.dynamicSmemBytes = F_SMEM_TOTAL; cfg.stream = stream;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int mcl = max_clusters[dev][ntile].load();
  if (mcl == 0) {
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(refiner_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, F_SMEM_TOTAL));
    cfg.gridDim = dim3(2 * ntile);
    SSLAM_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&mcl, refiner_fused_kernel, &cfg));
    SSLAM_REQUIRE(mcl >= 1, SSLAM_EUNSUPPORTED, "refiner: no cluster of %d CTAs fits on this device", 2 * ntile);
    max_clusters[dev][ntile].store(mcl);
  }
  int groups = mcl < nsp ? mcl : nsp;
  const int cap = 160 / (2 * ntile);
  if (groups > cap) groups = cap;
  int S = g_refiner_fused;                                       // 1..F_MAX_SLOTS (sslam_debug_refiner_fused)
  const int per_cluster = (nsp + groups - 1) / groups;
  if (S > per_cluster) S = per_cluster;                          // short inputs: no unused scratch slots
  const size_t srows = (size_t)groups * S * 2 * BM;
  SSLAM_REQUIRE(srows <= fused_scratch_rows(rows, Hd), SSLAM_EWORKSPACE, "refiner: fused scratch too small");

  // scratch: h pair, u pair (core-matrix layout, see fused_epilogue_tile: per 128-row strip
  // [column / 8][row / 8][row % 8][column % 8], columns padded to whole 64-column blocks), four partial-sum arrays
  const size_t hd_pad = (size_t)(Hd + F_BK - 1) / F_BK * F_BK;
  char* wp = reinterpret_cast<char*>(align_up(reinterpret_cast<uintptr_t>(scratch), 1024));
  auto take = [&](size_t bytes, size_t al) { char* q = wp; wp += align_up(bytes, al); return q; };
  Pair sh{reinterpret_cast<__half*>(take(srows * hd_pad * 4, 1024)), nullptr};
  sh.lo = sh.hi + SCR_PART;
  Pair su{reinterpret_cast<__half*>(take(srows * hd_pad * 4, 1024)), nullptr};
  su.lo = su.hi + SCR_PART;
  if (hd_pad != (size_t)Hd)     // the pad columns are multiplied (by zero weights): they must not hold NaN / Inf bit patterns
    SSLAM_CHECK_CUDA(cudaMemsetAsync(sh.hi, 0, 2 * align_up(srows * hd_pad * 4, 1024), stream));
  FusedParams fp = {};
  for (int i = 0; i < 2; ++i) {
    fp.st_sum[i] = reinterpret_cast<float*>(take((size_t)2 * ntile * srows * 4, 256));
    fp.st_sq[i] = reinterpret_cast<float*>(take((size_t)2 * ntile * srows * 4, 256));
  }
  fp.rows = rows; fp.C = C; fp.Hd = Hd; fp.D = D; fp.L = L; fp.S = S; fp.groups = groups; fp.ntile = ntile;
  fp.s_hi[0] = sh.hi; fp.s_lo[0] = sh.lo; fp.s_hi[1] = su.hi; fp.s_lo[1] = su.lo; fp.raw = raw; fp.stat_stride = srows;

  FusedMaps m;
  int rc;
  if ((rc = make_tensor_map_2d(&m.a_hi[0], xs.hi, rows, C, BM, F_BK, 2, 128))) return rc;
  if ((rc = make_tensor_map_2d(&m.a_lo[0], xs.lo, rows, C, BM, F_BK, 2, 128))) return rc;
  // scratch arrays as flat memory: rows of 1 KB (256 words), a stage = 32 consecutive rows, no swizzle
  const uint64_t flat_rows = srows * hd_pad * 4 / 1024;
  if ((rc = make_tensor_map_2d(&m.a_hi[1], sh.hi, flat_rows, 256, F_STAGE_BYTES / 1024, 256, 4, 0))) return rc;
  if ((rc = make_tensor_map_2d(&m.a_hi[2], su.hi, flat_rows, 256, F_STAGE_BYTES / 1024, 256, 4, 0))) return rc;
  m.a_lo[1] = m.a_hi[1]; m.a_lo[2] = m.a_hi[2];                  // (unused: one request fetches both parts)
  for (int l = 0; l < F_MAX_LAYERS; ++l) {
    const int ll = l < L ? l : L - 1;                            // unused entries alias a valid map
    const int K = ll == 0 ? C : Hd, N = ll == L - 1 ? D : Hd;
    if ((rc = make_tensor_map_2d(&m.w_hi[l], layers[ll].w.hi, N, K, 64, BK, 2))) return rc;
    if ((rc = make_tensor_map_2d(&m.w_lo[l], layers[ll].w.lo, N, K, 64, BK, 2))) return rc;
    fp.bias[l] = layers[ll].bias;
    fp.s1[l] = layers[ll].s1;
  }
  cfg.gridDim = dim3(2u * ntile * groups);
  SSLAM_LAUNCH(KK_GEMM, stream, cudaLaunchKernelEx(&cfg, refiner_fused_kernel, m, fp));
  return SSLAM_OK;
}

// packed weights: per Linear the fp16 hi then lo copies of the [out, in] matrix; the LayerNorm-fed
// ones (fc1, fc2 of every block) are stored folded and followed by s1[out], c0[out] (fp32)
size_t pair_bytes(size_t n) { return 2 * align_up(n * 2, 256); }
size_t vec_bytes(size_t n) { return 2 * align_up(n * 4, 256); }
size_t packed_total(int C, int Hd, int D, int blocks) {
  return pair_bytes((size_t)Hd * C) + (size_t)blocks * 2 * (pair_bytes((size_t)Hd * Hd) + vec_bytes(Hd)) +
         pair_bytes((size_t)D * Hd);
}

}  // namespace
}  // namespace sslam

using namespace sslam;

// params order (device pointers, fp32):
//   [0] input_proj.weight [Hd,C]   [1] input_proj.bias [Hd]
//   per block b (8 entries from 2 + 8b): norm1.weight, norm1.bias, fc1.weight [Hd,Hd], fc1.bias,
//                                        norm2.weight, norm2.bias, fc2.weight [Hd,Hd], fc2.bias
//   [2+8*blocks] output_proj.weight [D,Hd]   [3+8*blocks] output_proj.bias [D]
extern "C" size_t sslam_refiner_packed_bytes(int C, int Hd, int D, int blocks) {
  if (C <= 0 || Hd <= 0 || D <= 0 || blocks < 0) return 0;
  return packed_total(C, Hd, D, blocks) + 256;
}

extern "C" int sslam_refiner_pack_weights(const float* const* params, int C, int Hd, int D, int blocks,
                                          void* packed, size_t packed_bytes, void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  SSLAM_REQUIRE(params && packed, SSLAM_EINVAL, "refiner_pack: null pointer");
  SSLAM_REQUIRE(C % 8 == 0 && Hd % 8 == 0 && D % 4 == 0, SSLAM_EUNSUPPORTED,
                "refiner: C and hidden must be multiples of 8, D of 4 (C=%d Hd=%d D=%d)", C, Hd, D);
  SSLAM_REQUIRE(packed_bytes >= sslam_refiner_packed_bytes(C, Hd, D, blocks), SSLAM_EWORKSPACE,
                "refiner_pack: packed buffer too small");
  char* w = static_cast<char*>(packed);
  auto take_pair = [&](size_t n) {
    Pair d{reinterpret_cast<__half*>(w), reinterpret_cast<__half*>(w + align_up(n * 2, 256))};
    w += pair_bytes(n);
    return d;
  };
  if ((rc = launch_split(params[0], take_pair((size_t)Hd * C), (size_t)Hd * C, stream))) return rc;
  for (int b = 0; b < blocks; ++b) {
    const float* const* bp = params + 2 + 8 * b;
    for (int half = 0; half < 2; ++half) {                 // fc1 folded with norm1, fc2 with norm2
      Pair d = take_pair((size_t)Hd * Hd);
      float* s1 = reinterpret_cast<float*>(w);
      float* c0 = reinterpret_cast<float*>(w + align_up((size_t)Hd * 4, 256));
      w += vec_bytes(Hd);
      SSLAM_LAUNCH(KK_SPLIT, stream,
                   fold_ln_kernel<<<(Hd + 7) / 8, 256, 0, stream>>>(bp[4 * half + 2], bp[4 * half], bp[4 * half + 1],
                                                                    bp[4 * half + 3], Hd, Hd, d.hi, d.lo, s1, c0));
    }
  }
  return launch_split(params[2 + 8 * blocks], take_pair((size_t)D * Hd), (size_t)D * Hd, stream);
}

extern "C" size_t sslam_refiner_workspace_bytes(int rows, int C, int Hd, int D, int blocks) {
  (void)blocks;
  if (rows <= 0) return 0;
  const size_t r = (size_t)rows;
  // pairs (4 B/element): x [r,C]; h_a, h_b, u [r,Hd];  fp32 raw [r,D];  3 sets of partial row sums
  return (r * C + 3 * r * Hd + r * D) * 4 + 6 * (size_t)stat_parts_of(Hd) * stat_stride_of(rows) * 4 + 16 * 256 +
         fused_scratch_bytes(rows, Hd);
}

extern "C" int sslam_refiner_forward_f32(const float* const* params, const void* packed, const float* x,
                                         const void* x_hi, const void* x_lo,
                                         int rows, int C, int Hd, int D, int blocks, float eps_norm,
                                         float* out_f32, void* out_bf16, void* out_hi, void* out_lo,
                                         void* ws, size_t ws_bytes, void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  SSLAM_REQUIRE(rows >= 0, SSLAM_EINVAL, "refiner: negative rows");
  if (rows == 0) return SSLAM_OK;
  SSLAM_REQUIRE(params && packed && (x || (x_hi && x_lo)) && ws && (out_f32 || out_bf16 || out_hi), SSLAM_EINVAL,
                "refiner: null pointer");
  SSLAM_REQUIRE(C % 8 == 0 && Hd % 8 == 0 && D % 4 == 0 && Hd <= MAX_N && D <= MAX_N, SSLAM_EUNSUPPORTED,
                "refiner: C and hidden must be multiples of 8, D of 4, hidden and D <= 1024 (C=%d Hd=%d D=%d)", C, Hd, D);
  SSLAM_REQUIRE(!x || (reinterpret_cast<uintptr_t>(x) & 15) == 0, SSLAM_EINVAL, "refiner: x must be 16-byte aligned");
  SSLAM_REQUIRE(ws_bytes >= sslam_refiner_workspace_bytes(rows, C, Hd, D, blocks), SSLAM_EWORKSPACE,
                "refiner: workspace %zu < %zu", ws_bytes, sslam_refiner_workspace_bytes(rows, C, Hd, D, blocks));
  const size_t r = (size_t)rows;
  char* wp = static_cast<char*>(ws);
  auto take_pair = [&](size_t n) {
    Pair q{reinterpret_cast<__half*>(wp), reinterpret_cast<__half*>(wp + align_up(n * 2, 256))};
    wp += pair_bytes(n);
    return q;
  };
  auto take_stats = [&]() {
    const size_t n = (size_t)stat_parts_of(Hd) * stat_stride_of(rows);
    RowStats st{reinterpret_cast<float*>(wp), reinterpret_cast<float*>(wp) + n, 0};
    wp += 2 * n * 4;
    return st;
  };
  Pair xs = take_pair(r * C), h_a = take_pair(r * Hd), h_b = take_pair(r * Hd), u = take_pair(r * Hd);
  RowStats st_a = take_stats(), st_b = take_stats(), st_u = take_stats();
  float* raw = reinterpret_cast<float*>(wp);
  char* fused_scratch = reinterpret_cast<char*>(align_up(reinterpret_cast<uintptr_t>(wp) + r * D * 4, 256));
  const char* pk = static_cast<const char*>(packed);
  auto next_w = [&](size_t n) {
    Pair q{reinterpret_cast<__half*>(const_cast<char*>(pk)),
           reinterpret_cast<__half*>(const_cast<char*>(pk) + align_up(n * 2, 256))};
    pk += pair_bytes(n);
    return q;
  };
  const Pair none{nullptr, nullptr};
  const RowStats no_stats{nullptr, nullptr, 0};

  if (x) {
    if ((rc = launch_split(x, xs, r * C, stream))) return rc;
  } else {                                                                // pair written by the gather kernel
    xs.hi = static_cast<__half*>(const_cast<void*>(x_hi));
    xs.lo = static_cast<__half*>(const_cast<void*>(x_lo));
  }
  if (fused_eligible(C, Hd, D, blocks)) {
    // one persistent launch for all layers (refiner_fused_kernel); activations stay in L2
    FusedLayer layers[F_MAX_LAYERS];
    int nl = 0;
    layers[nl++] = FusedLayer{next_w((size_t)Hd * C), params[1], nullptr};
    for (int b = 0; b < blocks; ++b)
      for (int half = 0; half < 2; ++half) {
        const Pair wl = next_w((size_t)Hd * Hd);
        const float* s1 = reinterpret_cast<const float*>(pk);
        const float* c0 = reinterpret_cast<const float*>(pk + align_up((size_t)Hd * 4, 256));
        pk += vec_bytes(Hd);
        layers[nl++] = FusedLayer{wl, c0, s1};
      }
    layers[nl++] = FusedLayer{next_w((size_t)D * Hd), params[3 + 8 * blocks], nullptr};
    if ((rc = launch_fused(xs, layers, rows, C, Hd, D, blocks, raw, fused_scratch, stream))) return rc;
    return sslam_l2norm_rows(raw, rows, D, eps_norm, out_f32, out_bf16, out_hi, out_lo, stream_);   // :86
  }
  Pair w = next_w((size_t)Hd * C);                                        // descriptor_refiner.py:76
  if ((rc = launch_gemm(xs, w, rows, Hd, C, params[1], no_stats, nullptr, none, 1, nullptr, h_a,
                        blocks ? &st_a : nullptr, stream)))
    return rc;
  Pair h_cur = h_a, h_nxt = h_b;
  RowStats st_cur = st_a, st_nxt = st_b;
  for (int b = 0; b < blocks; ++b) {                                      // :79-80, :108-126
    // fc1( LN1(h) ) + ReLU, LayerNorm folded into the weights and the epilogue
    w = next_w((size_t)Hd * Hd);
    const float* s1 = reinterpret_cast<const float*>(pk);
    const float* c0 = reinterpret_cast<const float*>(pk + align_up((size_t)Hd * 4, 256));
    pk += vec_bytes(Hd);
    if ((rc = launch_gemm(h_cur, w, rows, Hd, Hd, c0, st_cur, s1, none, 1, nullptr, u, &st_u, stream))) return rc;
    // fc2( LN2(u) ) + identity, ReLU
    w = next_w((size_t)Hd * Hd);
    s1 = reinterpret_cast<const float*>(pk);
    c0 = reinterpret_cast<const float*>(pk + align_up((size_t)Hd * 4, 256));
    pk += vec_bytes(Hd);
    const bool last = (b == blocks - 1);
    if ((rc = launch_gemm(u, w, rows, Hd, Hd, c0, st_u, s1, h_cur, 1, nullptr, h_nxt, last ? nullptr : &st_nxt,
                          stream)))
      return rc;
    Pair tp = h_cur; h_cur = h_nxt; h_nxt = tp;
    RowStats ts = st_cur; st_cur = st_nxt; st_nxt = ts;
  }
  w = next_w((size_t)D * Hd);                                             // :83
  if ((rc = launch_gemm(h_cur, w, rows, D, Hd, params[3 + 8 * blocks], no_stats, nullptr, none, 0, raw, none,
                        nullptr, stream)))
    return rc;
  return sslam_l2norm_rows(raw, rows, D, eps_norm, out_f32, out_bf16, out_hi, out_lo, stream_);   // :86
}

extern "C" int sslam_refiner_range_check(void* stream_) {
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  unsigned int h = 0;
  SSLAM_CHECK_CUDA(cudaMemcpyFromSymbolAsync(&h, sslam::g_refiner_status, sizeof(h), 0, cudaMemcpyDeviceToHost, stream));
  SSLAM_CHECK_CUDA(cudaStreamSynchronize(stream));
  if (h) {
    const unsigned int zero = 0;
    SSLAM_CHECK_CUDA(cudaMemcpyToSymbolAsync(sslam::g_refiner_status, &zero, sizeof(zero), 0, cudaMemcpyHostToDevice, stream));
    SSLAM_CHECK_CUDA(cudaStreamSynchronize(stream));
    SSLAM_REQUIRE(false, SSLAM_ERANGE,
                  "refiner: an activation reached the fp16 range (|x| >= 65504, or NaN / inf) in the f16x3 arithmetic");
  }
  return SSLAM_OK;
}

// Debug aid for tests / tools: 0 = one GEMM launch per layer (gemm_pair_kernel); 1..4 = the layer-fused
// kernel with that many strip pairs per chunk (default 3).  Other values are clamped to 0..4.
extern "C" void sslam_debug_refiner_fused(int mode) {
  sslam::g_refiner_fused = mode < 0 ? 0 : (mode > sslam::F_MAX_SLOTS ? sslam::F_MAX_SLOTS : mode);
}

// Debug aid for tools/: host-mapped buffer (device pointer) that receives watchdog records of this
// translation unit's kernels; see tc_common.cuh.
extern "C" int sslam_debug_watchdog_gemm(unsigned long long* buf) {
  return (int)cudaMemcpyToSymbol(sslam::tc::g_watchdog_buf, &buf, sizeof(buf));
}
