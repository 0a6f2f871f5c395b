// Tensor-core similarity with the top-2 / argmax epilogue fused in: tcgen05.mma accumulating in
// TMEM, operands staged by TMA into swizzled shared memory, mbarrier pipelines, no similarity
// matrix in HBM.  Two kernels:
//
//   match_res_kernel<F16X3 | BF16>  (further down) — the production path.  CTA pairs (cta_group::2,
//       M = 256): each CTA keeps its 128-row strip of set 1 resident in shared memory and half of
//       every streamed B tile; rank 0 issues the MMAs of both.
//         SSLAM_SIM_F16X3 : "fp32 mode".  x ~= hi + lo * 2^-11 with hi, lo fp16 (22 significant
//                           bits); S = Ah.Bh + 2^-11 (Ah.Bl + Al.Bh) on kind::f16 MMAs.
//         SSLAM_SIM_BF16  : S = A.B^T on bf16 copies, fp32 accumulate.
//   match_tc_kernel<TF32X3>  (directly below) — the streaming single-CTA kernel, kept as the
//       cross-check of f16x3: hi = tf32(x), lo = tf32(x - hi), kind::tf32 (half the tensor rate,
//       twice the operand bytes).
//
// In both split modes the tensor core adds into its fp32 accumulator with truncation, so the
// 2^-11-sized cross terms are kept in their OWN TMEM accumulator and added to the Ah.Bh accumulator
// once, in the epilogue, with a round-to-nearest FMA; measured on B200 this takes the error from
// ~3e-6 to < 1e-6.  The dropped Al.Bl term is <= 2^-22 |a||b|.  Against the exact-mode kernel
// (match_f32.cu) decisions are identical except for similarity near-ties (< 1e-6), which the parity
// tests count.
//
// Roles in both kernels: warp 0 TMA producer, warp 1 MMA issuer (one elected thread), the remaining
// warps epilogue (thread = row: running (best, index, second) per row; column argmax per 32-row
// chunk merged across strips by a 64-bit atomicMax on (ordered value << 32 | ~row)).  Two TMEM
// accumulator sets let the epilogue of tile t overlap the MMAs of tile t+1.
//
// match_tc_kernel: a work item is one 128-row strip of one pair; the CTA walks the 128-wide column
// tiles, loading the A and B tiles of every term per k-block; four epilogue warps transpose each
// 32x32 chunk through padded shared memory for the column scan (redux.sync cost ~16k cycles/tile).
#include "tc_common.cuh"

#include <mutex>

namespace sslam {

using namespace tc;

namespace {

constexpr int BM = 128, BN = 128;
constexpr int BLOCK_BYTES = BM * 128;            // one operand tile: 128 rows x 128 bytes of K
constexpr int NUM_THREADS = 192;
constexpr int TP_LD = 36;                        // padded row length (floats) of the transpose tile

template <int MODE> struct Cfg;
template <> struct Cfg<SSLAM_SIM_TF32X3> {
  static constexpr int TERMS = 2, STAGES = 3, BK = 32, ACC_COLS = 2 * BN, TMEM_COLS = 512;
  static constexpr bool TF32 = true;
  static constexpr uint32_t FMT = FMT_TF32;
  static constexpr float CROSS_SCALE = 1.0f;
};
struct TcParams {
  const int32_t* pair_index;
  int P, N, M, D;
  int32_t* nn12;
  float* best12;
  float* second12;
  u64* colkeys;
};

template <int MODE>
struct SmemLayout {
  using C = Cfg<MODE>;
  static constexpr int STAGE_BYTES = 2 * C::TERMS * BLOCK_BYTES;     // A terms then B terms
  static constexpr int OPERANDS = C::STAGES * STAGE_BYTES;
  static constexpr int COLPART = 2 * 4 * BN * 8;                     // [acc][warp][col] u64
  static constexpr int TRANSP = 4 * 32 * TP_LD * 4;                  // [warp][32 rows][TP_LD] fp32
  static constexpr int BARS = (2 * C::STAGES + 4) * 8 + 16;
  static constexpr int TOTAL = OPERANDS + COLPART + TRANSP + BARS + 1024;   // + alignment slack
};

template <int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
match_tc_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                TcParams p) {
  using C = Cfg<MODE>;
  using L = SmemLayout<MODE>;
  extern __shared__ unsigned char smem_raw[];
  // 1024-byte alignment for SWIZZLE_128B; offset arithmetic keeps the pointer in the shared space
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* operands = smem;
  u64* colpart = reinterpret_cast<u64*>(smem + L::OPERANDS);
  float* transp = reinterpret_cast<float*>(smem + L::OPERANDS + L::COLPART);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::OPERANDS + L::COLPART + L::TRANSP);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int strips = (p.N + BM - 1) / BM;
  const int nitems = strips * p.P;             // persistent: items blockIdx.x, +gridDim.x, ...
  const int ntile = (p.M + BN - 1) / BN;
  const int nkb = (p.D + C::BK - 1) / C::BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (elect_one()) {
      prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmB_hi);
      if (C::TERMS == 2) { prefetch_tensormap(&tmA_lo); prefetch_tensormap(&tmB_lo); }
      int stage = 0; uint32_t phase = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
      const int pair = item / strips;
      int ia = pair, ib = pair;
      if (p.pair_index) { ia = p.pair_index[2 * pair]; ib = p.pair_index[2 * pair + 1]; }
      const int a_row = ia * p.N + (item - pair * strips) * BM;   // row coordinate in the [F*N, D] map
      const int b_row0 = ib * p.M;
      for (int ct = 0; ct < ntile; ++ct) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          unsigned char* st = operands + stage * L::STAGE_BYTES;
          mbar_arrive_expect_tx(&full[stage], L::STAGE_BYTES);
          const int kc = kb * C::BK;
          tma_load_2d(st, &tmA_hi, &full[stage], kc, a_row);
          if (C::TERMS == 2) tma_load_2d(st + BLOCK_BYTES, &tmA_lo, &full[stage], kc, a_row);
          tma_load_2d(st + C::TERMS * BLOCK_BYTES, &tmB_hi, &full[stage], kc, b_row0 + ct * BN);
          if (C::TERMS == 2)
            tma_load_2d(st + 3 * BLOCK_BYTES, &tmB_lo, &full[stage], kc, b_row0 + ct * BN);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (elect_one()) {
      const uint32_t idesc = make_instr_desc(C::FMT, BM, BN);
      int stage = 0; uint32_t phase = 0;
      const int my_tiles = ((nitems - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x) * ntile;
      for (int tc = 0; tc < my_tiles; ++tc) {                   // tc: running tile count of this CTA
        const int acc = tc & 1;
        const uint32_t acc_phase = (tc >> 1) & 1;
        mbar_wait(&tempty[acc], acc_phase ^ 1);                 // epilogue drained this accumulator
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * C::ACC_COLS;          // Ah.Bh (or the only term)
        const uint32_t tmem_s = tmem_d + BN;                            // cross terms (tf32x3)
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full[stage], phase);                       // TMA bytes have landed
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(operands + stage * L::STAGE_BYTES);
          const uint64_t a_hi = make_smem_desc_sw128(sa);
          const uint64_t a_lo = make_smem_desc_sw128(sa + BLOCK_BYTES);
          const uint64_t b_hi = make_smem_desc_sw128(sa + C::TERMS * BLOCK_BYTES);
          const uint64_t b_lo = make_smem_desc_sw128(sa + 3 * BLOCK_BYTES);
#pragma unroll
          for (int k = 0; k < 128 / 32; ++k) {                  // 32 bytes of K per instruction
            const uint64_t adv = (uint64_t)(k * 32 >> 4);
            const uint32_t first = (kb | k) ? 1u : 0u;
            if (C::TERMS == 2) {
              umma_ss<C::TF32>(tmem_s, a_lo + adv, b_hi + adv, idesc, first);
              umma_ss<C::TF32>(tmem_s, a_hi + adv, b_lo + adv, idesc, 1u);
              umma_ss<C::TF32>(tmem_d, a_hi + adv, b_hi + adv, idesc, first);
            } else {
              umma_ss<C::TF32>(tmem_d, a_hi + adv, b_hi + adv, idesc, first);
            }
          }
          tcgen05_commit(&empty[stage]);                        // smem stage reusable when MMAs retire
          if (kb == nkb - 1) tcgen05_commit(&tfull[acc]);       // accumulator complete
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ================================ epilogue (warps 2..5) ================================
    const int q = warp & 3;                                     // TMEM lane quarter of this warp
    const int ew = warp - 2;                                    // 0..3, slot in colpart
    const int et = threadIdx.x - 64;                            // 0..127
    float* tp = transp + ew * 32 * TP_LD;
    const float NEG_INF = __int_as_float(0xff800000);
    int tc = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int pair = item / strips;
    const int row0 = (item - pair * strips) * BM;
    const int grow = row0 + q * 32 + lane;                      // row of this thread inside the pair
    const bool row_ok = grow < p.N;
    int nvalid = p.N - (row0 + q * 32);                         // valid rows of this warp (uniform)
    nvalid = nvalid < 0 ? 0 : (nvalid > 32 ? 32 : nvalid);
    float best = NEG_INF, second = NEG_INF;
    int bidx = 0x7fffffff;
    for (int ct = 0; ct < ntile; ++ct, ++tc) {
      const int acc = tc & 1;
      const uint32_t acc_phase = (tc >> 1) & 1;
      mbar_wait(&tfull[acc], acc_phase);
      tcgen05_fence_after();
      u64* cp = colpart + (acc * 4 + ew) * BN;
      const int c0 = ct * BN;
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * C::ACC_COLS + ch * 32;
        tmem_ld_32x32(taddr, r);
        if (C::TERMS == 2) {
          uint32_t rs[32];
          tmem_ld_32x32(taddr + BN, rs);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j)
            r[j] = __float_as_uint(__fmaf_rn(__uint_as_float(rs[j]), C::CROSS_SCALE, __uint_as_float(r[j])));
        } else {
          tmem_ld_wait();
        }
        // row: columns arrive in ascending order, strict '>' keeps the lowest index (branch-free)
        const int gc0 = c0 + ch * 32;
        if (gc0 + 32 > p.M) {                                   // ragged last tile (warp-uniform)
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (gc0 + j >= p.M) r[j] = 0xff800000u;             // -inf never wins, never second
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float v = __uint_as_float(r[j]);
          const bool gt = v > best;
          second = gt ? best : fmaxf(second, v);
          bidx = gt ? (gc0 + j) : bidx;
          best = gt ? v : best;
        }
        // column: transpose the 32x32 chunk through smem, lane j scans column j top-down
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<uint4*>(tp + lane * TP_LD + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
        __syncwarp();
        float cm = 0.f;
        int cr = -1;
        if (nvalid == 32) {                                     // two independent chains, merged
          float m0 = tp[lane], m1 = tp[16 * TP_LD + lane];
          int r0 = 0, r1 = 16;
#pragma unroll
          for (int rr = 1; rr < 16; ++rr) {                     // rows ascending: lowest row wins ties
            const float v0 = tp[rr * TP_LD + lane], v1 = tp[(16 + rr) * TP_LD + lane];
            if (v0 > m0) { m0 = v0; r0 = rr; }
            if (v1 > m1) { m1 = v1; r1 = 16 + rr; }
          }
          cm = m0; cr = r0;
          if (m1 > m0) { cm = m1; cr = r1; }
        } else {
          for (int rr = 0; rr < nvalid; ++rr) {
            const float v = tp[rr * TP_LD + lane];
            if (cr < 0 || v > cm) { cm = v; cr = rr; }
          }
        }
        cp[ch * 32 + lane] = (cr >= 0) ? pack_key(cm, (u32)(row0 + q * 32 + cr)) : 0ull;
      }
      // accumulator fully read: hand it back to the MMA warp
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      // merge the four warps' column results and publish
      named_bar_sync(1, 128);
      {
        const u64* base = colpart + acc * 4 * BN;
        u64 k = base[et];
#pragma unroll
        for (int w = 1; w < 4; ++w) { u64 o = base[w * BN + et]; k = o > k ? o : k; }
        if (c0 + et < p.M && k) atomicMax(p.colkeys + (size_t)pair * p.M + c0 + et, k);
      }
    }
    if (row_ok) {
      const size_t o = (size_t)pair * p.N + grow;
      p.nn12[o] = bidx; p.best12[o] = best; p.second12[o] = second;
    }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// A-resident variant (f16x3 and bf16: the 128-row strip of set 1 fits in shared memory).
//
// The streaming kernel above re-reads the A strip for every column tile, so each 128x128 tile pulls
// 2 x TERMS x 16 KB per k-block through L2 — at 148 SMs that is the L2 slice throughput limit
// (~42 B/cycle/SM measured), not the tensor pipe.  Here the strip is loaded once per work item and
// stays in shared memory (per-k-block barriers, so the next item's strip streams in while the last
// tile of the current item is still being multiplied); only B tiles stream, in 16 KB stages.
// f16x3 issues three M=256 (cta_group::2) MMAs per k-step — A_lo x B_hi and A_hi x B_lo into the
// cross-term accumulator (TMEM columns [128,256)), A_hi x B_hi into the main one ([0,128)); each CTA
// of the pair holds half of every B tile.  Eight epilogue warps (two per TMEM lane quarter, 64 columns
// each) keep the epilogue under the MMA time of a tile.
template <int MODE> struct RCfg;
template <> struct RCfg<SSLAM_SIM_F16X3> {
  static constexpr int TERMS = 2, B_BK = 64, B_SWZ = 128, B_STAGES = 4, ACC_COLS = 2 * BN, TMEM_COLS = 512;
  static constexpr uint32_t FMT = FMT_F16;
  static constexpr float CROSS_SCALE = 1.0f / 2048.0f;
};
template <> struct RCfg<SSLAM_SIM_BF16> {
  static constexpr int TERMS = 1, B_BK = 64, B_SWZ = 128, B_STAGES = 6, ACC_COLS = BN, TMEM_COLS = 256;
  static constexpr uint32_t FMT = FMT_BF16;
  static constexpr float CROSS_SCALE = 1.0f;
};
constexpr int R_EPI_WARPS = 8;
constexpr int R_THREADS = 64 + 32 * R_EPI_WARPS;
constexpr int R_MAX_KB = 4;                      // D <= 256: four 64-element k-blocks of A
constexpr int R_UNIT = 16;                       // columns per epilogue step

template <int MODE>
struct RSmem {
  using C = RCfg<MODE>;
  static constexpr int A_BYTES = R_MAX_KB * C::TERMS * BLOCK_BYTES;
  static constexpr int B_TILE = (BN / 2) * C::B_BK * 2;              // one term of one stage: this CTA's 64 of the tile's 128 rows
  static constexpr int B_STAGE = C::TERMS * B_TILE;                  // hi then lo
  static constexpr int OPERANDS = A_BYTES + C::B_STAGES * B_STAGE;
  static constexpr int COLPART = 2 * 4 * BN * 8;                     // [acc][lane quarter][col] u64
  static constexpr int TRANSP = R_EPI_WARPS * 32 * R_UNIT * 4;       // [warp][32 rows][16] fp32, swizzled
  static constexpr int ROWMERGE = 2 * BM * 3 * 4;                    // [item parity][row][best, idx, second]
  static constexpr int BARS = (2 * C::B_STAGES + 2 * R_MAX_KB + 4) * 8 + 16;
  static_assert(C::B_BK == 64, "the pair kernel stages whole 64-element k-blocks");
  static constexpr int TOTAL = OPERANDS + COLPART + TRANSP + ROWMERGE + BARS + 1024;
};

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(R_THREADS, 1)
match_res_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                 const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                 TcParams p) {
  using C = RCfg<MODE>;
  using L = RSmem<MODE>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* a_res = smem;
  unsigned char* b_stages = smem + L::A_BYTES;
  u64* colpart = reinterpret_cast<u64*>(smem + L::OPERANDS);
  float* transp = reinterpret_cast<float*>(smem + L::OPERANDS + L::COLPART);
  float* rowmerge = reinterpret_cast<float*>(smem + L::OPERANDS + L::COLPART + L::TRANSP);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::OPERANDS + L::COLPART + L::TRANSP + L::ROWMERGE);
  uint64_t* full = bars;
  uint64_t* empty = full + C::B_STAGES;
  uint64_t* afull = empty + C::B_STAGES;
  uint64_t* aempty = afull + R_MAX_KB;
  uint64_t* tfull = aempty + R_MAX_KB;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA pair (cta_group::2): the two CTAs own two adjacent 128-row strips of the SAME pair and share
  // every MMA (M = 256); each holds its own strip resident and HALF of every B tile (64 of its 128
  // rows), so the B stream per SM — shared-memory writes, L2 traffic and, for a given number of
  // bytes in flight, pipeline depth — is half of what a single CTA needs.  Work item of the pair =
  // (pair of sets, strip pair); rank 0 issues the MMAs.
  const uint32_t rank = cluster_ctarank();
  const int strips = (p.N + BM - 1) / BM;
  const int strips2 = (strips + 1) / 2;
  const int nitems = strips2 * p.P;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int ntile = (p.M + BN - 1) / BN;
  const int nkb = (p.D + 63) / 64;                                    // k-blocks = B stages per tile

  if (threadIdx.x == 0) {
    // full / afull live in the leader: its expect_tx arrival + one arrival of the peer's producer, so
    // that both producers take part in every use (no producer can be overtaken by two phases)
    for (int s = 0; s < C::B_STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], 1); }
    for (int k = 0; k < R_MAX_KB; ++k) { mbar_init(&afull[k], 2); mbar_init(&aempty[k], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * R_EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, C::TMEM_COLS);
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================ TMA producer (both CTAs) ================================
    if (elect_one()) {
      prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmB_hi);
      if (C::TERMS == 2) { prefetch_tensormap(&tmA_lo); prefetch_tensormap(&tmB_lo); }
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int item = pair_id; item < nitems; item += npairs, ++it) {
        const int pair = item / strips2;
        int ia = pair, ib = pair;
        if (p.pair_index) { ia = p.pair_index[2 * pair]; ib = p.pair_index[2 * pair + 1]; }
        // an odd strip count leaves the last item of a pair with one real strip: the other CTA runs
        // the same loop on rows past the set (masked in the epilogue)
        const int a_row = ia * p.N + (2 * (item - pair * strips2) + (int)rank) * BM;
        const int b_row0 = ib * p.M + (int)rank * (BN / 2);
        for (int ct = 0; ct < ntile; ++ct) {
          for (int kb = 0; kb < nkb; ++kb) {
            if (ct == 0) {                                      // this item's A k-block (own strip)
              mbar_wait(&aempty[kb], (uint32_t)(it & 1) ^ 1u);  // last tile of the previous item done with it
              const uint32_t afull_leader = mapa_u32(smem_u32(&afull[kb]), 0);
              if (rank == 0) mbar_arrive_expect_tx(&afull[kb], 2u * C::TERMS * BLOCK_BYTES);
              else mbar_arrive_cluster(afull_leader);
              tma_load_2d_pair(a_res + (kb * C::TERMS) * BLOCK_BYTES, &tmA_hi, afull_leader, kb * 64, a_row);
              if (C::TERMS == 2)
                tma_load_2d_pair(a_res + (kb * C::TERMS + 1) * BLOCK_BYTES, &tmA_lo, afull_leader, kb * 64, a_row);
            }
            mbar_wait(&empty[stage], phase ^ 1);
            unsigned char* st = b_stages + stage * L::B_STAGE;
            const uint32_t full_leader = mapa_u32(smem_u32(&full[stage]), 0);
            if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2u * L::B_STAGE);
            else mbar_arrive_cluster(full_leader);
            tma_load_2d_pair(st, &tmB_hi, full_leader, kb * 64, b_row0 + ct * BN);
            if (C::TERMS == 2) tma_load_2d_pair(st + L::B_TILE, &tmB_lo, full_leader, kb * 64, b_row0 + ct * BN);
            if (++stage == C::B_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
      // producer tail: the last empty / aempty arrivals are asynchronous tensor-core commits into this
      // CTA's shared memory; drain them before the CTA may exit
      for (int i = 0; i < C::B_STAGES; ++i) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (++stage == C::B_STAGES) { stage = 0; phase ^= 1; }
      }
      if (it > 0)
        for (int kb = 0; kb < nkb; ++kb) mbar_wait(&aempty[kb], (uint32_t)(it & 1) ^ 1u);
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA) ================================
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = make_instr_desc(C::FMT, 2 * BM, BN);      // M = 256 across the pair
      int stage = 0; uint32_t phase = 0;
      int tc = 0, it = 0;
      for (int item = pair_id; item < nitems; item += npairs, ++it) {
        for (int ct = 0; ct < ntile; ++ct, ++tc) {
          const int acc = tc & 1;
          mbar_wait(&tempty[acc], (((uint32_t)tc >> 1) & 1u) ^ 1u);
          tcgen05_fence_after();
          const uint32_t tmem_d = tmem_base + acc * C::ACC_COLS;
          for (int kb = 0; kb < nkb; ++kb) {
            if (ct == 0) mbar_wait(&afull[kb], (uint32_t)(it & 1));
            mbar_wait(&full[stage], phase);
            tcgen05_fence_after();
            const uint32_t sa = smem_u32(a_res + (kb * C::TERMS) * BLOCK_BYTES);
            const uint32_t sb = smem_u32(b_stages + stage * L::B_STAGE);
            const uint64_t a_hi = make_smem_desc_sw128(sa);
            const uint64_t a_lo = make_smem_desc_sw128(sa + BLOCK_BYTES);
            const uint64_t b_hi = make_smem_desc_sw128(sb);
            const uint64_t b_lo = make_smem_desc_sw128(sb + L::B_TILE);
#pragma unroll
            for (int k = 0; k < 4; ++k) {                       // 16 elements = 32 bytes of K per instruction
              const uint64_t adv = (uint64_t)(k * 32 >> 4);
              const uint32_t first = (kb | k) ? 1u : 0u;
              if (C::TERMS == 2) {
                umma_ss_pair(tmem_d + BN, a_lo + adv, b_hi + adv, idesc, first);
                umma_ss_pair(tmem_d + BN, a_hi + adv, b_lo + adv, idesc, 1u);
              }
              umma_ss_pair(tmem_d, a_hi + adv, b_hi + adv, idesc, first);
            }
            tcgen05_commit_pair(&empty[stage], 3);
            if (ct == ntile - 1) tcgen05_commit_pair(&aempty[kb], 3);
            if (kb == nkb - 1) tcgen05_commit_pair(&tfull[acc], 3);
            if (++stage == C::B_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else {
    // ================================ epilogue (warps 2..9) ================================
    const int q = warp & 3;                                     // TMEM lane quarter of this warp
    const int ew = warp - 2;
    const int half = ew >> 2;                                   // which 64 columns of every tile
    const int et = threadIdx.x - 64;                            // 0..255
    float* tp = transp + ew * 32 * R_UNIT;
    const int sc = lane & 15, srh = lane >> 4;                  // column scan: column / row parity
    const float NEG_INF = __int_as_float(0xff800000);
    int tc = 0, it = 0;
    const uint32_t tempty_leader0 = mapa_u32(smem_u32(&tempty[0]), 0);
    const uint32_t tempty_leader1 = mapa_u32(smem_u32(&tempty[1]), 0);
    for (int item = pair_id; item < nitems; item += npairs, ++it) {
      const int pair = item / strips2;
      const int row0 = (2 * (item - pair * strips2) + (int)rank) * BM;
      const int grow = row0 + q * 32 + lane;
      const bool row_ok = grow < p.N;
      int nvalid = p.N - (row0 + q * 32);
      nvalid = nvalid < 0 ? 0 : (nvalid > 32 ? 32 : nvalid);
      float best = NEG_INF, second = NEG_INF;
      int bidx = 0x7fffffff;
      for (int ct = 0; ct < ntile; ++ct, ++tc) {
        const int acc = tc & 1;
        mbar_wait(&tfull[acc], ((uint32_t)tc >> 1) & 1u);
        tcgen05_fence_after();
        u64* cp = colpart + (acc * 4 + q) * BN;
        const int c0 = ct * BN;
        // Units of 16 columns, software pipelined: the TMEM loads of unit u+1 are in flight while
        // unit u is reduced.
        //   row   : running (best, second) by value only — a pairwise max/min tree over the 16 new
        //           values, three FMNMX per node; the index is looked up (first column equal to the
        //           new maximum) only in the units that raise a row's maximum, which become rare
        //           after the first tiles of an item;
        //   column: the 32x16 chunk is transposed through shared memory (16-byte pieces XOR-swizzled
        //           by row pair: the row-wise stores and the column-wise loads are both conflict
        //           free); lane (c, parity) loads its 16 rows at once and reduces them as two
        //           independent chains, the two parities are merged with one shuffle.
        uint32_t r[R_UNIT], rs[R_UNIT];
        {
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * C::ACC_COLS + half * 64;
          tmem_ld_32x16(taddr, r);
          if (C::TERMS == 2) tmem_ld_32x16(taddr + BN, rs);
        }
#pragma unroll
        for (int un = 0; un < 64 / R_UNIT; ++un) {
          const int col0 = half * 64 + un * R_UNIT;
          const int gc0 = c0 + col0;
          float v[R_UNIT];
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < R_UNIT; ++j)
            v[j] = C::TERMS == 2 ? __fmaf_rn(__uint_as_float(rs[j]), C::CROSS_SCALE, __uint_as_float(r[j]))
                                 : __uint_as_float(r[j]);
          if (un + 1 < 64 / R_UNIT) {
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * C::ACC_COLS + col0 + R_UNIT;
            tmem_ld_32x16(taddr, r);
            if (C::TERMS == 2) tmem_ld_32x16(taddr + BN, rs);
          }
          if (gc0 + R_UNIT > p.M) {                             // ragged last tile (warp-uniform)
#pragma unroll
            for (int j = 0; j < R_UNIT; ++j)
              if (gc0 + j >= p.M) v[j] = NEG_INF;               // never wins, never second
          }
          // ---- row top-2 (values), index on demand
          {
            float tb[R_UNIT / 2], ts[R_UNIT / 2];
#pragma unroll
            for (int j = 0; j < R_UNIT / 2; ++j) {
              tb[j] = fmaxf(v[2 * j], v[2 * j + 1]);
              ts[j] = fminf(v[2 * j], v[2 * j + 1]);
            }
#pragma unroll
            for (int w = R_UNIT / 4; w >= 1; w >>= 1) {
#pragma unroll
              for (int j = 0; j < w; ++j) {
                const float lo = fminf(tb[2 * j], tb[2 * j + 1]);
                ts[j] = fmaxf(fmaxf(ts[2 * j], ts[2 * j + 1]), lo);
                tb[j] = fmaxf(tb[2 * j], tb[2 * j + 1]);
              }
            }
            const float ub = tb[0];
            second = fmaxf(fmaxf(second, ts[0]), fminf(best, ub));
            if (ub > best) {                                    // strict: an earlier column keeps ties
              best = ub;
              int f = R_UNIT - 1;
#pragma unroll
              for (int j = R_UNIT - 2; j >= 0; --j) f = (v[j] == ub) ? j : f;   // first column equal to ub
              bidx = gc0 + f;
            }
          }
          // ---- column argmax over the warp's 32 rows
          if (nvalid < 32 && !row_ok) {
#pragma unroll
            for (int j = 0; j < R_UNIT; ++j) v[j] = NEG_INF;    // rows past N never win a column
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < R_UNIT / 4; ++j)
            *reinterpret_cast<float4*>(tp + lane * R_UNIT + ((j ^ ((lane >> 1) & 3)) << 2)) =
                make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          __syncwarp();
          float cv[16];
#pragma unroll
          for (int rr = 0; rr < 16; ++rr)
            cv[rr] = tp[(2 * rr + srh) * R_UNIT + ((((sc >> 2) ^ (rr & 3))) << 2) + (sc & 3)];
          float m0 = cv[0], m1 = cv[8];
          int r0 = 0, r1 = 8;
#pragma unroll
          for (int rr = 1; rr < 8; ++rr) {                      // rows ascending: lowest row wins ties
            if (cv[rr] > m0) { m0 = cv[rr]; r0 = rr; }
            if (cv[8 + rr] > m1) { m1 = cv[8 + rr]; r1 = 8 + rr; }
          }
          float cm = m0;
          int cr = r0;
          if (m1 > m0) { cm = m1; cr = r1; }
          cr = 2 * cr + srh;
          {
            const float om = __shfl_xor_sync(0xffffffffu, cm, 16);
            const int orow = __shfl_xor_sync(0xffffffffu, cr, 16);
            if (om > cm || (om == cm && orow < cr)) { cm = om; cr = orow; }
          }
          if (srh == 0) cp[col0 + sc] = (nvalid > 0) ? pack_key(cm, (u32)(row0 + q * 32 + cr)) : 0ull;
        }
        // accumulator fully read: hand it back to the MMA warp
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(acc ? tempty_leader1 : tempty_leader0);
        // merge the four lane quarters' column results and publish
        named_bar_sync(1, 32 * R_EPI_WARPS);
        if (et < BN) {
          const u64* base = colpart + acc * 4 * BN;
          u64 k = base[et];
#pragma unroll
          for (int w = 1; w < 4; ++w) { u64 o = base[w * BN + et]; k = o > k ? o : k; }
          if (c0 + et < p.M && k) atomicMax(p.colkeys + (size_t)pair * p.M + c0 + et, k);
        }
      }
      // merge the two column halves of every row (half 1 hands its state to half 0)
      float* rm = rowmerge + (it & 1) * (BM * 3) + (q * 32 + lane) * 3;
      if (half == 1) { rm[0] = best; rm[1] = __int_as_float(bidx); rm[2] = second; }
      named_bar_sync(1, 32 * R_EPI_WARPS);
      if (half == 0 && row_ok) {
        const float ob = rm[0], os = rm[2];
        const int oi = __float_as_int(rm[1]);
        // second = second largest of the union, duplicates of the maximum count
        const float lo_best = fminf(best, ob);
        float sec = fmaxf(fmaxf(second, os), lo_best);
        if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
        const size_t o = (size_t)pair * p.N + grow;
        p.nn12[o] = bidx; p.best12[o] = best; p.second12[o] = sec;
      }
    }
  }
  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, C::TMEM_COLS);
}

// fp32 -> (tf32 hi, tf32 lo) split of a descriptor bank
__global__ void split_tf32_kernel(const float4* __restrict__ src, float4* __restrict__ hi,
                                  float4* __restrict__ lo, size_t n4) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) {
    float4 x = __ldg(src + i), h, l;
    h.x = to_tf32_rna(x.x); h.y = to_tf32_rna(x.y); h.z = to_tf32_rna(x.z); h.w = to_tf32_rna(x.w);
    l.x = to_tf32_rna(__fsub_rn(x.x, h.x)); l.y = to_tf32_rna(__fsub_rn(x.y, h.y));
    l.z = to_tf32_rna(__fsub_rn(x.z, h.z)); l.w = to_tf32_rna(__fsub_rn(x.w, h.w));
    hi[i] = h; lo[i] = l;
  }
}

// fp32 -> (fp16 hi, fp16 lo * 2^11) split of a descriptor bank
__global__ void split_f16_kernel(const float4* __restrict__ src, uint2* __restrict__ hi,
                                 uint2* __restrict__ lo, size_t n4) {
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

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
std::once_flag g_encode_once;

}  // namespace

namespace tc {
int make_tensor_map_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols,
                       uint32_t box_rows, uint32_t box_cols, int elem_bytes, int swizzle_bytes) {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  SSLAM_REQUIRE(g_encode != nullptr, SSLAM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  if (swizzle_bytes < 0) return SSLAM_OK;                      // entry-point resolution only
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  // 2-byte elements are moved as opaque 16-bit words (bf16 and fp16 alike)
  CUresult r = g_encode(map, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                        2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                             : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SSLAM_REQUIRE(r == CUDA_SUCCESS, SSLAM_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return SSLAM_OK;
}
// NHWC tensor [B,H,W,C] (2-byte elements) as a 4-D map with a {box_c, box_w, box_h, 1} box and
// 128-byte swizzle: box_c * 2 bytes = 128, so a box lands in shared memory as box_h*box_w rows of 128
// bytes — the K-major SWIZZLE_128B operand tile whose rows are the pixels of a (box_h x box_w) window.
// Coordinates may be negative / beyond the image: those elements are zero-filled (convolution padding).
int make_tensor_map_nhwc(CUtensorMap* map, const void* base, uint64_t B, uint64_t H, uint64_t W, uint64_t C,
                         uint32_t box_h, uint32_t box_w, uint32_t box_c) {
  int rc = make_tensor_map_2d(nullptr, nullptr, 0, 0, 0, 0, 0, -1);      // resolves the driver entry point only
  if (rc) return rc;
  cuuint64_t dims[4] = {C, W, H, B};
  cuuint64_t strides[3] = {C * 2, W * C * 2, H * W * C * 2};
  cuuint32_t box[4] = {box_c, box_w, box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SSLAM_REQUIRE(r == CUDA_SUCCESS, SSLAM_ECUDA, "cuTensorMapEncodeTiled (NHWC) failed with CUresult %d", (int)r);
  return SSLAM_OK;
}
}  // namespace tc

namespace {

// When bank2 lies inside / directly after bank1 on a frame boundary (sequence mode: bank2 =
// bank1 + one frame) the two banks are split once, over their union.
struct BankPlan {
  bool shared;           // one split region serves both banks
  size_t frames_a, frames_b, off_b_frames;
};

BankPlan plan_banks(const float* b1, int F1, const float* b2, int F2, int N, int M, int D) {
  BankPlan pl{false, (size_t)F1, (size_t)F2, 0};
  if (N != M) return pl;
  const size_t frame = (size_t)N * D;
  const float* end1 = b1 + (size_t)F1 * frame;
  if (b2 >= b1 && b2 <= end1 && ((size_t)(b2 - b1) % frame) == 0) {
    pl.shared = true;
    pl.off_b_frames = (size_t)(b2 - b1) / frame;
    size_t uni = pl.off_b_frames + (size_t)F2;
    pl.frames_a = uni > (size_t)F1 ? uni : (size_t)F1;
  }
  return pl;
}

}  // namespace

size_t match_tc_extra_workspace(int P, int N, int M, int D, int dtype, int F1, int F2) {
  (void)P;
  if (dtype != SSLAM_SIM_TF32X3 && dtype != SSLAM_SIM_F16X3) return 0;
  // worst case: both banks split separately (hi + lo each); fp16 pairs take half the bytes
  const size_t e = dtype == SSLAM_SIM_F16X3 ? 2 : 4;
  return 2 * align_up((size_t)F1 * N * D * e, 256) + 2 * align_up((size_t)F2 * M * D * e, 256) + 1024;
}

template <int MODE>
static int launch_tc(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi,
                     const CUtensorMap& b_lo, const TcParams& tp, cudaStream_t stream) {
  using L = SmemLayout<MODE>;
  static DeviceOnce once;
  if (once.first_use()) {
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(match_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          L::TOTAL));
  }
  const int strips = (tp.N + BM - 1) / BM;
  SSLAM_LAUNCH(KK_MATCH_TC, stream,
               match_tc_kernel<MODE><<<strips * tp.P, NUM_THREADS, L::TOTAL, stream>>>(a_hi, a_lo, b_hi, b_lo, tp));
  return SSLAM_OK;
}

template <int MODE>
static int launch_res(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi,
                      const CUtensorMap& b_lo, const TcParams& tp, cudaStream_t stream) {
  using L = RSmem<MODE>;
  static DeviceOnce once;
  if (once.first_use()) {
    SSLAM_CHECK_CUDA(cudaFuncSetAttribute(match_res_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          L::TOTAL));
  }
  const int items = ((((tp.N + BM - 1) / BM) + 1) / 2) * tp.P;      // (pair of sets, strip pair)
  const int pairs = items < num_sms() / 2 ? items : num_sms() / 2;
  const int grid = 2 * pairs;                                      // persistent: one CTA pair per TPC
  SSLAM_LAUNCH(KK_MATCH_TC, stream,
               match_res_kernel<MODE><<<grid, R_THREADS, L::TOTAL, stream>>>(a_hi, a_lo, b_hi, b_lo, tp));
  return SSLAM_OK;
}

int match_top2_tc(const void* bank1, const void* bank1_lo, int F1, const void* bank2, const void* bank2_lo,
                  int F2, const int32_t* pair_index,
                  int dtype, int P, int N, int M, int D, int32_t* nn12, float* best12, float* second12,
                  u64* colkeys, void* ws_extra, size_t ws_extra_bytes, cudaStream_t stream) {
  TcParams tp;
  tp.pair_index = pair_index; tp.P = P; tp.N = N; tp.M = M; tp.D = D;
  tp.nn12 = nn12; tp.best12 = best12; tp.second12 = second12; tp.colkeys = colkeys;
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
  int rc;
  if (dtype == SSLAM_SIM_BF16) {
    SSLAM_REQUIRE(D % 8 == 0, SSLAM_EUNSUPPORTED, "match(bf16): D=%d must be a multiple of 8", D);
    if ((rc = make_tensor_map_2d(&a_hi, bank1, (uint64_t)F1 * N, D, BM, 64, 2))) return rc;
    if ((rc = make_tensor_map_2d(&b_hi, bank2, (uint64_t)F2 * M, D, BN / 2, 64, 2))) return rc;   // half tile per CTA
    a_lo = a_hi; b_lo = b_hi;
    return launch_res<SSLAM_SIM_BF16>(a_hi, a_lo, b_hi, b_lo, tp, stream);
  }
  // ---- split modes: the fp32 banks are split into hi / lo (tf32 pairs or fp16 pairs)
  const bool f16 = (dtype == SSLAM_SIM_F16X3);
  const size_t e = f16 ? 2 : 4;
  SSLAM_REQUIRE(!f16 || D % 8 == 0, SSLAM_EUNSUPPORTED, "match(f16x3): D=%d must be a multiple of 8", D);
  if (f16 && bank1_lo && bank2_lo) {
    // banks arrive as fp16 (hi, lo) pairs (written by the L2-normalisation kernel): nothing to split
    const uint64_t rows2p = (uint64_t)F2 * M;
    if ((rc = make_tensor_map_2d(&a_hi, bank1, (uint64_t)F1 * N, D, BM, 64, 2))) return rc;
    if ((rc = make_tensor_map_2d(&a_lo, bank1_lo, (uint64_t)F1 * N, D, BM, 64, 2))) return rc;
    if ((rc = make_tensor_map_2d(&b_hi, bank2, rows2p, D, BN / 2, 64, 2))) return rc;        // half tile per CTA
    if ((rc = make_tensor_map_2d(&b_lo, bank2_lo, rows2p, D, BN / 2, 64, 2))) return rc;
    return launch_res<SSLAM_SIM_F16X3>(a_hi, a_lo, b_hi, b_lo, tp, stream);
  }
  SSLAM_REQUIRE(ws_extra_bytes >= match_tc_extra_workspace(P, N, M, D, dtype, F1, F2), SSLAM_EWORKSPACE,
                "match(split): workspace too small");
  const float* f1 = static_cast<const float*>(bank1);
  const float* f2 = static_cast<const float*>(bank2);
  char* w = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws_extra) + 1023) & ~(uintptr_t)1023);
  const BankPlan pl = plan_banks(f1, F1, f2, F2, N, M, D);
  const size_t n1 = pl.frames_a * (size_t)N * D;
  char* h1 = w;
  char* l1 = w + align_up(n1 * e, 256);
  const int sms = num_sms();
  auto split = [&](const float* src, char* hi, char* lo, size_t n) -> int {
    if (f16)
      SSLAM_LAUNCH(KK_SPLIT, stream,
                   split_f16_kernel<<<sms * 8, 256, 0, stream>>>(reinterpret_cast<const float4*>(src),
                                                                 reinterpret_cast<uint2*>(hi),
                                                                 reinterpret_cast<uint2*>(lo), n / 4));
    else
      SSLAM_LAUNCH(KK_SPLIT, stream,
                   split_tf32_kernel<<<sms * 8, 256, 0, stream>>>(reinterpret_cast<const float4*>(src),
                                                                  reinterpret_cast<float4*>(hi),
                                                                  reinterpret_cast<float4*>(lo), n / 4));
    return SSLAM_OK;
  };
  if ((rc = split(f1, h1, l1, n1))) return rc;
  char *h2, *l2;
  if (pl.shared) {
    h2 = h1 + pl.off_b_frames * (size_t)N * D * e;
    l2 = l1 + pl.off_b_frames * (size_t)N * D * e;
  } else {
    const size_t n2 = (size_t)F2 * M * D;
    char* w2 = w + 2 * align_up(n1 * e, 256);
    h2 = w2;
    l2 = w2 + align_up(n2 * e, 256);
    if ((rc = split(f2, h2, l2, n2))) return rc;
  }
  const uint64_t rows2 = (uint64_t)F2 * M;
  if (f16) {
    // A strip resident (128-byte swizzled 64-element k-blocks), B streamed in 32-element / 64-byte
    // swizzled stages
    if ((rc = make_tensor_map_2d(&a_hi, h1, (uint64_t)F1 * N, D, BM, 64, 2))) return rc;
    if ((rc = make_tensor_map_2d(&a_lo, l1, (uint64_t)F1 * N, D, BM, 64, 2))) return rc;
    if ((rc = make_tensor_map_2d(&b_hi, h2, rows2, D, BN / 2, 64, 2))) return rc;            // half tile per CTA
    if ((rc = make_tensor_map_2d(&b_lo, l2, rows2, D, BN / 2, 64, 2))) return rc;
    return launch_res<SSLAM_SIM_F16X3>(a_hi, a_lo, b_hi, b_lo, tp, stream);
  }
  if ((rc = make_tensor_map_2d(&a_hi, h1, (uint64_t)F1 * N, D, BM, 32, 4))) return rc;
  if ((rc = make_tensor_map_2d(&a_lo, l1, (uint64_t)F1 * N, D, BM, 32, 4))) return rc;
  if ((rc = make_tensor_map_2d(&b_hi, h2, rows2, D, BN, 32, 4))) return rc;
  if ((rc = make_tensor_map_2d(&b_lo, l2, rows2, D, BN, 32, 4))) return rc;
  return launch_tc<SSLAM_SIM_TF32X3>(a_hi, a_lo, b_hi, b_lo, tp, stream);
}

}  // namespace sslam
