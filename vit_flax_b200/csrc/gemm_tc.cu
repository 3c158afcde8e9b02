// gemm_tc.cu -- K3: persistent, warp-specialised tcgen05 GEMM (bf16 or fp16 operands; E4M3 for the fp8 precision's
// to_qkv / FeedForward, kind::f8f6f4 on 128-element k-blocks) with fused epilogues.  acc[M,N] = A[M,K] x Wt[N,K]^T,
// fp32 accumulation in TMEM.
//
// Replaces every flax `nn.Dense` on the hot path (vit.py:48,51,68,82,147,165) together with what
// follows it in the reference: bias add, tanh-GELU (vit.py:49), the Residual add (vit.py:39),
// cls/pos-embedding placement (vit.py:151-153).
//
// Structure (one CTA per SM, 12 warps):
//   warp 0  lane 0 : TMA producer  (A box 128x64, Wt box 256x64, SWIZZLE_128B)
//   warp 1  lane 0 : tcgen05.mma issuer, M=128 N=256 K=16, 4 per smem stage
//   warp 2         : TMEM allocator (512 columns = 2 accumulator stages)
//   warps 4..11    : epilogue, two groups of 4 warps (one warp per TMEM lane quarter);
//                    group g owns the 128-byte-wide column slabs s = g, g+2, ... of the tile:
//                    tcgen05.ld -> fused math -> swizzled smem slab -> TMA store
//                    (16-bit outputs, fp32 head) or TMA reduce-add into the fp32 residual
//                    stream (x += acc + bias happens in L2; the SM never reads x).
// Tile modes (template kCG): 2 = CTA pair (cluster of 2, `cta_group::2`) on a 256x256 tile -- each
// CTA loads its 128 rows of A and its 128-row half of Wt, only the leader issues MMAs -- is the
// production mode: the single-CTA 128x256 form (1) is smem-bandwidth bound at ~62 % tensor-pipe
// activity.  64 = single CTA on 128x64 tiles for problems of one or two row blocks; 4 = cluster of
// two pairs sharing a multicast weight tile (opt-in, profiles/r01_gemm.md).
// Pipelines: smem ring (3 / 5 / 6 stages for modes 1 / 2,4 / 64; full/empty mbarriers) between TMA
// and MMA; TMEM double buffer (tfull/tempty mbarriers) between MMA and epilogue, so the epilogue of
// tile i overlaps the MMAs of tile i+1; two slab buffers per epilogue group so a slab drains while
// the next is filled.  Dropout (template kDrop) is applied in the epilogues that have an
// nn.Dropout behind them in the reference (ptx.cuh: dropout4).
//
// LayerNorm fold (PreNorm, vit.py:31; SURVEY.md H4-ii): LN(x) W = rstd (x W') - rstd mean c + d with
// W' = diag(gamma) W, c = 1^T W', d = beta^T W (+ bias).  The GEMMs that PRODUCE the residual stream
// (TOKENS_LN, RESID_LN) also emit a 16-bit copy of the raw x and per-row partial sums (sum, sum of
// squares -- Flax's E[x^2] - E[x]^2 variance) of the fp32 values; the GEMMs that CONSUME a LayerNorm
// (LN_STORE_16 = to_qkv, LN_GELU_16 = FeedForward Dense_0) read the raw 16-bit x as A and apply the
// row statistics in their epilogue.  No stand-alone LayerNorm kernel runs between them.  RESID_LN has
// to see x_old in the SM (the plain RESID epilogue adds in L2 and never does): the epilogue groups pull
// the 128x32 fp32 slabs of x by TMA two slabs ahead into a ring of three buffers, add in place and
// TMA-store them back.  Statistics partials go to one slot per (n-tile, epilogue group) and are summed
// in slot order by the consumer: no atomics, bit-reproducible.
#include <cstdlib>

#include "common.h"
#include "ptx.cuh"

namespace vb {

namespace {

constexpr int BM = GEMM_BM, BN = GEMM_BN, BK = GEMM_BK;
constexpr int UMMA_K = 16;
constexpr int A_BYTES = BM * BK * 2;            // 16 KB: 128 rows of A per CTA
// kCG: 1 = one CTA per 128x256 tile; 2 = CTA pair (cta_group::2) per 256x256 tile; 4 = cluster of two
// pairs working on two vertically adjacent 256x256 tiles that share their weight tile: each CTA
// fetches a quarter of it and TMA-multicasts it to its opposite number in the other pair.
// kCG (tile mode): 1 = one CTA per 128x256 tile; 2 = CTA pair (cta_group::2) per 256x256 tile; 4 =
// cluster of two pairs sharing a multicast weight tile; 64 = one CTA per 128x64 tile (small problems:
// four times as many tiles, so a forward at batch 1..32 spreads over the SMs instead of 3..12 CTAs).
template <int kCG> struct Cfg {
  static constexpr int CL = kCG == 64 ? 1 : kCG;                // CTAs per cluster
  static constexpr int BN_ = kCG == 64 ? 64 : BN;               // tile columns
  static constexpr int MMA_CG = CL == 1 ? 1 : 2;                // tcgen05 cta_group
  static constexpr int STAGES = kCG == 64 ? 6 : (CL == 1 ? 3 : 5);
  static constexpr int B_ROWS = BN_ / MMA_CG;                   // rows of Wt in this CTA's smem
  static constexpr int B_LOAD_ROWS = BN_ / CL;                  // rows of Wt this CTA fetches
  static constexpr int B_BYTES = B_ROWS * BK * 2;               // 32 KB / 16 KB / 8 KB
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;         // 48 KB / 32 KB / 24 KB
  static constexpr int TILE_M = BM * MMA_CG;                    // 128 / 256
  static constexpr int PAIRS = kCG == 4 ? 2 : 1;                // tiles per cluster step
  static constexpr int TMEM_COLS = BN_ == 64 ? 128 : 512;       // two accumulator stages
};
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 128 + NUM_EPI_WARPS * 32;   // 384
constexpr int SLAB_BYTES = BM * 128;            // 128 rows x 128 B = 16 KB
// slab buffers per epilogue group: 2 (one drains while the next is filled); RESID_LN: a ring of 3 (x_old
// loads run two slabs ahead), paid for with one smem stage
template <int kEpi> __host__ __device__ constexpr int slabs_per_group() { return kEpi == VITB200_EPI_RESID_LN ? 3 : 2; }
template <int kCG, int kEpi> __host__ __device__ constexpr int num_stages() {
  return Cfg<kCG>::STAGES - (kEpi == VITB200_EPI_RESID_LN ? 1 : 0);
}
template <int kCG, int kEpi = VITB200_EPI_STORE_16> constexpr int smem_bytes() {
  return num_stages<kCG, kEpi>() * Cfg<kCG>::STAGE_BYTES + 2 * slabs_per_group<kEpi>() * SLAB_BYTES + 1024 /*align*/ +
         256 /*barriers*/;
}

__device__ __forceinline__ float gelu_tanh_fast(float x) {
  // 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))  -- nn.gelu default (vit.py:49)
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * x * fmaf(k1 * x, x, 1.0f);
  return 0.5f * x * (1.0f + tanh_approx(u));
}

// The same on two values at a time (fp32x2: one issue slot for two lanes of FFMA / FMUL -- the GELU epilogue of
// FeedForward Dense_0 is the most instruction-heavy one and sits next to the MMA time of its K = dim tiles):
// u = x (k0 + k0 k1 x^2), gelu = hx + hx tanh(u) with hx = 0.5 x.
__device__ __forceinline__ unsigned long long gelu_tanh_fast2(unsigned long long x2) {
  const unsigned long long kA = pack_f32x2(0.7978845608028654f * 0.044715f, 0.7978845608028654f * 0.044715f);
  const unsigned long long kB = pack_f32x2(0.7978845608028654f, 0.7978845608028654f);
  const unsigned long long half2 = pack_f32x2(0.5f, 0.5f);
  const unsigned long long t2 = mul_f32x2(x2, x2);
  const unsigned long long u2 = mul_f32x2(fma_f32x2(t2, kA, kB), x2);
  float u0, u1;
  unpack_f32x2(u2, u0, u1);
  const unsigned long long th2 = pack_f32x2(tanh_approx(u0), tanh_approx(u1));
  const unsigned long long hx2 = mul_f32x2(x2, half2);
  return fma_f32x2(th2, hx2, hx2);
}

// kMN (weight gradients, dW = X^T dY): both operands are read MN-major straight from the row-major
// activations -- tmA over X [K rows, M cols], tmB over dY [K rows, N cols], boxes of 64 rows x 64
// columns -- so the K dimension of the GEMM is the ROW index and no transposed copy is needed.  A
// stage then holds, per operand, one 8 KB box per 64-column atom (LBO = 8 KB between atoms, 1 KB
// between 8-row groups); rows past K are zero-filled by TMA.
template <int kEpi, int kDT, int kCG, bool kDrop, bool kMN = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA,
               const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC,
               const float* __restrict__ bias, void* __restrict__ Cout,
               int M, int N, int K, const float* __restrict__ aux, int tpi, int dbg, Dropout drop, int cls_off,
               const float* __restrict__ cls, LnFold ln, const float* __restrict__ wscale) {
  // fp8 precision: E4M3 operands, k-blocks of 128 elements (still 128 B per row: the stage layout, boxes, barriers and
  // descriptors are those of the 16-bit form), the accumulator scaled per column by wscale; 16-bit outputs are fp16
  constexpr bool kF8 = (kDT == DT_E4M3);
  constexpr int kODT = kF8 ? DT_F16 : kDT;
  constexpr int KB = kF8 ? 128 : BK;                          // elements per k-block
  static_assert(!kF8 || (!kMN && !kDrop), "E4M3 operands: K-major, no dropout");
  constexpr bool kOut8 = (kEpi == VITB200_EPI_BIAS_GELU_E4M3);   // E4M3 output, 64-byte slab rows (64 columns)
  constexpr bool kOut16 = (kEpi == VITB200_EPI_STORE_16 || kEpi == VITB200_EPI_BIAS_GELU_16 || kEpi == VITB200_EPI_BIAS_16 ||
                           kEpi == VITB200_EPI_BIAS_PRE_GELU_16 || kEpi == VITB200_EPI_LN_STORE_16 ||
                           kEpi == VITB200_EPI_LN_GELU_16);
  constexpr bool kLnIn = (kEpi == VITB200_EPI_LN_STORE_16 || kEpi == VITB200_EPI_LN_GELU_16);   // A = raw x, LayerNorm applied here
  constexpr bool kLnOut = (kEpi == VITB200_EPI_RESID_LN || kEpi == VITB200_EPI_TOKENS_LN);      // also emits x16 + row statistics
  constexpr bool kLoadX = (kEpi == VITB200_EPI_RESID_LN);                                       // x_old comes in by TMA
  constexpr bool kTokens = (kEpi == VITB200_EPI_TOKENS_F32 || kEpi == VITB200_EPI_TOKENS_LN);
  constexpr int SPG = slabs_per_group<kEpi>();
  constexpr bool kDual = (kEpi == VITB200_EPI_BIAS_PRE_GELU_16);   // two outputs per slab: pre-activation and GELU
  constexpr bool kDirect = (kEpi == VITB200_EPI_PATCH_F32);   // row-remapped output: plain stores
  constexpr int SLAB_COLS = (kOut16 || kOut8) ? 64 : 32;      // 128 B (E4M3: 64 B) of output per row
  constexpr int SLABS_PER_TILE = Cfg<kCG>::BN_ / SLAB_COLS;
  constexpr int STAGES = num_stages<kCG, kEpi>(), B_BYTES = Cfg<kCG>::B_BYTES;
  constexpr int STAGE_BYTES = Cfg<kCG>::STAGE_BYTES, TILE_M = Cfg<kCG>::TILE_M;
  constexpr int MMA_CG = Cfg<kCG>::MMA_CG, PAIRS = Cfg<kCG>::PAIRS, CL = Cfg<kCG>::CL;
  constexpr int BN = Cfg<kCG>::BN_, TMEM_COLS = Cfg<kCG>::TMEM_COLS;   // shadow the 256-column default
  // crank: rank in the cluster; rank: 0 = leader of its CTA pair (issues the MMAs), 1 = peer;
  // pair: which of the cluster's tiles this CTA works on
  const uint32_t crank = CL == 1 ? 0u : cluster_ctarank();
  const uint32_t rank = crank & 1u, pair = crank >> 1;
  const uint32_t lead = crank & ~1u;                 // cluster rank of this pair's leader
  const int tile0 = int(blockIdx.x) / CL;            // cluster index
  const int tile_step = int(gridDim.x) / CL;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + STAGES * A_BYTES;
  const uint32_t sSlab = smem_base + STAGES * STAGE_BYTES;
  const uint32_t bars = sSlab + 2 * SPG * SLAB_BYTES;
  // barrier layout: full[STAGES] empty[STAGES] tfull[2] tempty[2] | tmem ptr | xfull[2 groups][3] (RESID_LN)
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bars + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bars + 8u * (2 * STAGES + 2 + s); };
  const uint32_t tmem_slot = bars + 8u * (2 * STAGES + 4);
  auto xfull_bar = [&](int g, int b) { return bars + 8u * (2 * STAGES + 5 + g * 3 + b); };
  uint32_t* tmem_slot_ptr =
      reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = ((M + TILE_M - 1) / TILE_M + PAIRS - 1) / PAIRS;   // cluster steps along M
  const int n_tiles = (N + BN - 1) / BN;
  const int num_kb = (K + KB - 1) / KB;
  // split-K (BIAS_RESID_F32 only, `tpi` carries the factor): split sp of a tile accumulates k-blocks
  // [sp * kb_per, min(num_kb, (sp + 1) * kb_per)) and reduce-adds its partial sum; split 0 adds the bias
  const int splits = (kEpi == VITB200_EPI_BIAS_RESID_F32 && tpi > 1) ? tpi : 1;
  const int kb_per = (num_kb + splits - 1) / splits;
  const int mn_tiles = m_tiles * n_tiles;
  const int num_tiles = mn_tiles * splits;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if constexpr (!kDirect) prefetch_tmap(&tmC);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);                       // pair: only the leader arrives (arms both CTAs' bytes)
      mbar_init(empty_bar(s), PAIRS);                  // cluster of 4: both pairs must have consumed the stage
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), NUM_EPI_WARPS * MMA_CG);   // pair: epilogue warps of both CTAs
    }
    if constexpr (kLoadX)
      for (int i = 0; i < 6; ++i) mbar_init(xfull_bar(i / 3, i % 3), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<MMA_CG>(tmem_slot, TMEM_COLS);
  tc_fence_before();
  if constexpr (CL != 1) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_launch_dependents();   // the next kernel's CTAs may take this SM as soon as this one leaves it
  pdl_wait();                // previous kernel complete: A, bias, the residual stream are final

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        const int sp = tile / mn_tiles, t2 = tile - sp * mn_tiles;
        const int m_blk = t2 / n_tiles, n_blk = t2 % n_tiles;
        const int kb0 = sp * kb_per, kb1 = min(num_kb, kb0 + kb_per);
        const int a_row = (m_blk * PAIRS + int(pair)) * TILE_M + int(rank) * BM;
        const int b_row = n_blk * BN + int(rank) * Cfg<kCG>::B_ROWS + int(pair) * Cfg<kCG>::B_LOAD_ROWS;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          if (dbg & 1) {   // timing experiment: no loads, the MMAs chew on stale smem
            if (rank == 0) mbar_arrive(full_bar(stage));
          } else if constexpr (CL == 1) {
            mbar_arrive_expect_tx(full_bar(stage), STAGE_BYTES);
            if constexpr (kMN) {
#pragma unroll
              for (int j = 0; j < BM / 64; ++j)
                tma_load_2d(sA + stage * A_BYTES + j * 8192, &tmA, full_bar(stage), a_row + j * 64, kb * BK);
#pragma unroll
              for (int j = 0; j < Cfg<kCG>::B_ROWS / 64; ++j)
                tma_load_2d(sB + stage * B_BYTES + j * 8192, &tmB, full_bar(stage), b_row + j * 64, kb * BK);
            } else {
              tma_load_2d(sA + stage * A_BYTES, &tmA, full_bar(stage), kb * KB, a_row);
              tma_load_2d(sB + stage * B_BYTES, &tmB, full_bar(stage), kb * KB, b_row);
            }
          } else {
            // Both CTAs' loads complete on the pair LEADER's full barrier (the MMA issuer waits there).
            // Only the leader arrives, arming the bytes of both CTAs: the peer's complete_tx may
            // land first (tx-count goes transiently negative) but the phase cannot complete
            // before the leader's arrival.  A remote arrive from the peer is not needed and its
            // cluster-scope release costs >1000 cycles per stage (profiles/r01_gemm_pair.md).
            const uint32_t lead_full = mapa_shared(full_bar(stage), lead);
            if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * STAGE_BYTES);
            if constexpr (kMN) {
              static_assert(!kMN || CL <= 2, "MN-major operands are not built for the multicast cluster");
#pragma unroll
              for (int j = 0; j < BM / 64; ++j)
                tma_load_2d_cg2(sA + stage * A_BYTES + j * 8192, &tmA, lead_full, a_row + j * 64, kb * BK);
#pragma unroll
              for (int j = 0; j < Cfg<kCG>::B_ROWS / 64; ++j)
                tma_load_2d_cg2(sB + stage * B_BYTES + j * 8192, &tmB, lead_full, b_row + j * 64, kb * BK);
            } else {
            tma_load_2d_cg2(sA + stage * A_BYTES, &tmA, lead_full, kb * KB, a_row);
            if constexpr (CL == 2) {
              tma_load_2d_cg2(sB + stage * B_BYTES, &tmB, lead_full, kb * KB, b_row);
            } else {
              // 64 of this CTA's 128 weight rows, delivered to the same smem offset here and in the
              // CTA of equal rank in the other pair; each destination signals its own pair leader.
              tma_load_2d_cg2_mc(sB + stage * B_BYTES + pair * (Cfg<kCG>::B_LOAD_ROWS * BK * 2), &tmB,
                                 lead_full, kb * BK, b_row, uint16_t(0x5u << rank));
            }
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only in pair mode) =====================
    if (rank == 0 && elect_one()) {
      constexpr uint32_t idesc = kF8 ? umma_idesc_e4m3(TILE_M, BN)
                                     : umma_idesc_16(TILE_M, BN, kDT == DT_F16 ? 0 : 1, kMN ? 1 : 0, kMN ? 1 : 0);
      const uint16_t pair_mask = uint16_t(0x3u << lead);               // both CTAs of this pair
      const uint16_t all_mask = uint16_t((1u << CL) - 1u);             // every CTA whose smem the stage's loads touch
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        if constexpr (CL != 1) mbar_wait_cluster(tempty_bar(acc), acc_phase ^ 1u);
        else mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        const int kb0 = (tile / mn_tiles) * kb_per, kb1 = min(num_kb, kb0 + kb_per);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t a0 = sA + stage * A_BYTES, b0 = sB + stage * B_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {   // E4M3: 4 x K = 32, the same 32-byte steps
            if constexpr (kF8)
              umma_f8_ss<MMA_CG>(d_tmem, umma_desc_k_sw128(a0 + k * UMMA_K * 2), umma_desc_k_sw128(b0 + k * UMMA_K * 2),
                                 idesc, (kb != kb0 || k != 0) ? 1u : 0u);
            else if constexpr (kMN)   // 16 K-rows of 128 B further per step
              umma_bf16_ss<MMA_CG>(d_tmem, umma_desc_mn_sw128_wide(a0 + k * UMMA_K * 128, 8192),
                                   umma_desc_mn_sw128_wide(b0 + k * UMMA_K * 128, 8192), idesc,
                                   (kb != kb0 || k != 0) ? 1u : 0u);
            else
            umma_bf16_ss<MMA_CG>(d_tmem, umma_desc_k_sw128(a0 + k * UMMA_K * 2),
                              umma_desc_k_sw128(b0 + k * UMMA_K * 2), idesc,
                              (kb != kb0 || k != 0) ? 1u : 0u);
          }
          // smem slot free (in both CTAs) once these MMAs retire
          if constexpr (CL != 1) umma_commit_cg2_mc(empty_bar(stage), all_mask);
          else umma_commit(empty_bar(stage));
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        // accumulator ready for the epilogue (of both CTAs)
        if constexpr (CL != 1) umma_commit_cg2_mc(tfull_bar(acc), pair_mask);
        else umma_commit(tfull_bar(acc));
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int ew = warp - 4;
    const int q = ew & 3;        // TMEM lane quarter this warp may access (== warp % 4)
    const int grp = ew >> 2;     // epilogue group: owns slabs grp, grp+2, ...
    const bool leader = (q == 0 && lane == 0);   // issues / waits the group's TMA stores
    const int lrow = q * 32 + lane;              // row inside the tile == TMEM lane
    int acc = 0;
    uint32_t acc_phase = 0;
    int buf = 0;
    // RESID_LN: the group's leader streams the x_old slabs in, two ahead of the slab being updated (ring of 3)
    int ld_tile = tile0, ld_s = grp, ld_issued = 0, x_used = 0;
    auto issue_x_load = [&]() {
      while (ld_tile < num_tiles) {
        if (ld_s < SLABS_PER_TILE && (ld_tile % n_tiles) * BN + ld_s * SLAB_COLS < N) break;
        ld_tile += tile_step;
        ld_s = grp;
      }
      if (ld_tile >= num_tiles) return;
      const int lm = ld_tile / n_tiles, lnb = ld_tile % n_tiles;      // RESID_LN never splits K: tile = m_blk * n_tiles + n_blk
      const int b = ld_issued % 3;
      mbar_arrive_expect_tx(xfull_bar(grp, b), SLAB_BYTES);
      tma_load_2d(sSlab + uint32_t(grp * SPG + b) * SLAB_BYTES, &tmC, xfull_bar(grp, b), lnb * BN + ld_s * SLAB_COLS,
                  (lm * PAIRS + int(pair)) * TILE_M + int(rank) * BM);
      ++ld_issued;
      ld_s += 2;
    };
    if constexpr (kLoadX) {
      if (leader) { issue_x_load(); issue_x_load(); }
    }
    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
      const int sp = tile / mn_tiles, t2 = tile - sp * mn_tiles;
      const int m_blk = t2 / n_tiles, n_blk = t2 % n_tiles;
      const int m_row0 = (m_blk * PAIRS + int(pair)) * TILE_M + int(rank) * BM;   // first output row of this CTA
      // LayerNorm of this thread's row of A (consumers): mean and rstd from the producer's partial sums, summed in
      // slot order (bit-reproducible); variance = E[x^2] - E[x]^2 like flax.linen.LayerNorm
      float ln_rstd = 0.f, ln_rm = 0.f;
      if constexpr (kLnIn) {
        if (m_row0 + lrow < M) {
          const float2* sp2 = ln.stats + int64_t(m_row0 + lrow) * ln.slots;
          float s1 = 0.f, s2 = 0.f;
          // two slots per 16-byte load (the slot count is even), up to eight slots in flight together: one L2 round trip
          // for the six slots of D = 768 instead of six dependent ones; the additions keep the slot order
          const float4* sp4 = reinterpret_cast<const float4*>(sp2);
          const int npair = (ln.slots & 1) ? 0 : ln.slots >> 1;
          if (ln.slots & 1) {   // an odd slot count (per-kernel entry point only): plain loop
            for (int i = 0; i < ln.slots; ++i) { const float2 v = __ldg(sp2 + i); s1 += v.x; s2 += v.y; }
          }
          for (int i = 0; i < npair; i += 4) {
            float4 a[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) a[u] = i + u < npair ? __ldg(sp4 + i + u) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (i + u < npair) { s1 += a[u].x; s2 += a[u].y; s1 += a[u].z; s2 += a[u].w; }
          }
          const float inv_d = 1.0f / float(K);
          const float mean = s1 * inv_d;
          ln_rstd = rsqrtf(fmaxf(s2 * inv_d - mean * mean, 0.f) + ln.eps);
          ln_rm = ln_rstd * mean;
        }
      }
      float st1 = 0.f, st2 = 0.f;       // producers: this thread's partial row sums over the group's slabs of the tile
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * BN);

      if constexpr (kDirect) {
        // ---- PATCH: row b*Np+t -> output row b*T+cls+t, + bias + pos_embedding[cls+t]; cls = 1 with a
        // class token in front of every image (ViT, vit.py:151-153), 0 without (SimpleViT) ----
        const int row = m_row0 + lrow;
        const bool row_ok = row < M;
        const int b = row / tpi, t = row - b * tpi;
        float* crow_base = reinterpret_cast<float*>(Cout) + (int64_t(b) * (tpi + cls_off) + cls_off + t) * N;
        const float* pos_row = aux + int64_t(cls_off + t) * N;
#pragma unroll 1
        for (int chunk = 0; chunk < BN / 64; ++chunk) {   // each group owns half of the tile's columns
          const int n0 = n_blk * BN + grp * (BN / 2) + chunk * 32;
          if (n0 >= N) break;                         // warp-uniform
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_row + uint32_t(grp * (BN / 2) + chunk * 32), r);
          tmem_ld_wait();
          if (row_ok) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (n0 + j * 4 < N) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + n0 + j * 4));
                const float4 p4 = __ldg(reinterpret_cast<const float4*>(pos_row + n0 + j * 4));
                float4 o;
                o.x = __uint_as_float(r[j * 4 + 0]) + b4.x + p4.x;
                o.y = __uint_as_float(r[j * 4 + 1]) + b4.y + p4.y;
                o.z = __uint_as_float(r[j * 4 + 2]) + b4.z + p4.z;
                o.w = __uint_as_float(r[j * 4 + 3]) + b4.w + p4.w;
                if constexpr (kDrop)   // emb dropout (vit.py:155) on the token stream, flat index = row * N + col
                  dropout4(drop, (int64_t(b) * (tpi + cls_off) + cls_off + t) * N + n0 + j * 4, o.x, o.y, o.z, o.w);
                *reinterpret_cast<float4*>(crow_base + n0 + j * 4) = o;
                if (cls != nullptr && t == 0) {
                  // the class token in front of image b (vit.py:151-153): row b*T = cls + pos_embedding[0],
                  // written by the thread that owns the image's first patch row
                  const float4 c4 = __ldg(reinterpret_cast<const float4*>(cls + n0 + j * 4));
                  const float4 q4 = __ldg(reinterpret_cast<const float4*>(aux + n0 + j * 4));
                  float4 z = make_float4(c4.x + q4.x, c4.y + q4.y, c4.z + q4.z, c4.w + q4.w);
                  const int64_t e0 = int64_t(b) * (tpi + 1) * N + n0 + j * 4;
                  if constexpr (kDrop) dropout4(drop, e0, z.x, z.y, z.z, z.w);
                  *reinterpret_cast<float4*>(reinterpret_cast<float*>(Cout) + e0) = z;
                }
              }
            }
          }
        }
      } else {
        // ---- slab epilogue: regs -> swizzled smem slab -> TMA store / reduce-add ----
#pragma unroll 1
        for (int s = grp; s < SLABS_PER_TILE; s += 2) {
          const int n0 = n_blk * BN + s * SLAB_COLS;
          if (n0 >= N || (dbg & 4)) break;             // uniform over the group
          const uint32_t slab = sSlab + uint32_t(grp * SPG + (kLoadX ? x_used % 3 : buf)) * SLAB_BYTES;
          if constexpr (kLoadX) {
            // the slab's x_old values have landed in the buffer (loaded two slabs ago, after the store that last
            // used the buffer had been read out)
            mbar_wait(xfull_bar(grp, x_used % 3), uint32_t(x_used / 3) & 1u);
          } else {
            // the slab buffer used two slabs ago must have been read out by its TMA store (dual output: both
            // buffers of the group are filled per slab, so every earlier store must have been read out)
            if (leader) { if constexpr (kDual) tma_store_wait_read<0>(); else tma_store_wait_read<1>(); }
            named_bar_sync(1 + grp, 128);
          }
          const uint32_t srow = slab + uint32_t(lrow) * 128u;
          const int sw = lrow & 7;
          // dual output: the GELU values go to the group's other slab buffer and leave `tpi` rows further down
          const uint32_t srow2 = sSlab + uint32_t(grp * 2 + (buf ^ 1)) * SLAB_BYTES + uint32_t(lrow) * 128u;
          if constexpr (kOut16) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t r[32];
              tmem_ld_32x32b_x32(t_row + uint32_t(s * SLAB_COLS + half * 32), r);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 4; ++j) {            // 8 columns -> one 16-byte chunk
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(r[j * 8 + e]);
                if constexpr (kF8) {   // STORE_16 (to_qkv): acc * the weight's column scale
                  const int nb = n0 + half * 32 + j * 8;
                  if (nb < N) {
                    const float4 w0 = __ldg(reinterpret_cast<const float4*>(wscale + nb));
                    const float4 w1 = __ldg(reinterpret_cast<const float4*>(wscale + nb + 4));
                    v[0] *= w0.x; v[1] *= w0.y; v[2] *= w0.z; v[3] *= w0.w;
                    v[4] *= w1.x; v[5] *= w1.y; v[6] *= w1.z; v[7] *= w1.w;
                  }
                }
                if constexpr (kEpi == VITB200_EPI_BIAS_16 || kDual) {   // pre-activation kept for the backward pass
                  const int nb = n0 + half * 32 + j * 8;
                  if (nb < N) {
                    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + nb));
                    const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + nb + 4));
                    v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
                    v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
                  }
                }
                if constexpr (kDual) {
                  // the GELU acts on the ROUNDED pre-activation, which is what the backward differentiates at
                  const int chunk2 = half * 4 + j;
                  const uint32_t q0 = pack2<kDT>(v[0], v[1]), q1 = pack2<kDT>(v[2], v[3]), q2 = pack2<kDT>(v[4], v[5]), q3 = pack2<kDT>(v[6], v[7]);
                  st_shared_v4(srow + (uint32_t(chunk2 ^ sw) << 4), q0, q1, q2, q3);
                  v[0] = to_f32<kDT>(uint16_t(q0 & 0xFFFFu)); v[1] = to_f32<kDT>(uint16_t(q0 >> 16));
                  v[2] = to_f32<kDT>(uint16_t(q1 & 0xFFFFu)); v[3] = to_f32<kDT>(uint16_t(q1 >> 16));
                  v[4] = to_f32<kDT>(uint16_t(q2 & 0xFFFFu)); v[5] = to_f32<kDT>(uint16_t(q2 >> 16));
                  v[6] = to_f32<kDT>(uint16_t(q3 & 0xFFFFu)); v[7] = to_f32<kDT>(uint16_t(q3 >> 16));
#pragma unroll
                  for (int e = 0; e < 8; ++e) v[e] = gelu_tanh_fast(v[e]);
                  if constexpr (kDrop) {   // FeedForward's first Dropout (vit.py:50)
                    const int64_t e0 = int64_t(m_row0 + lrow) * N + n0 + half * 32 + j * 8;
                    dropout4(drop, e0, v[0], v[1], v[2], v[3]);
                    dropout4(drop, e0 + 4, v[4], v[5], v[6], v[7]);
                  }
                  st_shared_v4(srow2 + (uint32_t(chunk2 ^ sw) << 4), pack2<kDT>(v[0], v[1]), pack2<kDT>(v[2], v[3]),
                               pack2<kDT>(v[4], v[5]), pack2<kDT>(v[6], v[7]));
                  continue;
                }
                if constexpr (kLnIn) {
                  // LayerNorm folded into the weights: y = rstd acc - rstd mean c + d  (d = beta W + bias), then GELU for FF
                  const int nb = n0 + half * 32 + j * 8;
                  float4 c0 = make_float4(0.f, 0.f, 0.f, 0.f), c1 = c0, d0 = c0, d1 = c0;
                  if (nb < N) {
                    c0 = __ldg(reinterpret_cast<const float4*>(ln.c + nb));
                    c1 = __ldg(reinterpret_cast<const float4*>(ln.c + nb + 4));
                    d0 = __ldg(reinterpret_cast<const float4*>(bias + nb));
                    d1 = __ldg(reinterpret_cast<const float4*>(bias + nb + 4));
                  }
                  const unsigned long long rs2 = pack_f32x2(ln_rstd, ln_rstd), nrm2 = pack_f32x2(-ln_rm, -ln_rm);
                  const float cc[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
                  const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
                  for (int e = 0; e < 8; e += 2) {
                    unsigned long long y2 = fma_f32x2(rs2, pack_f32x2(v[e], v[e + 1]),
                                                      fma_f32x2(nrm2, pack_f32x2(cc[e], cc[e + 1]), pack_f32x2(dd[e], dd[e + 1])));
                    if constexpr (kEpi == VITB200_EPI_LN_GELU_16) y2 = gelu_tanh_fast2(y2);
                    unpack_f32x2(y2, v[e], v[e + 1]);
                  }
                }
                if constexpr (kEpi == VITB200_EPI_BIAS_GELU_16) {
                  const int nb = n0 + half * 32 + j * 8;
                  float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
                  if (nb < N) {
                    b0 = __ldg(reinterpret_cast<const float4*>(bias + nb));
                    b1 = __ldg(reinterpret_cast<const float4*>(bias + nb + 4));
                  }
                  const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                  for (int e = 0; e < 8; e += 2)
                    unpack_f32x2(gelu_tanh_fast2(add_f32x2(pack_f32x2(v[e], v[e + 1]), pack_f32x2(bb[e], bb[e + 1]))), v[e], v[e + 1]);
                  if constexpr (kDrop) {   // FeedForward's first Dropout (vit.py:50), on the hidden activations
                    const int64_t e0 = int64_t(m_row0 + lrow) * N + nb;
                    dropout4(drop, e0, v[0], v[1], v[2], v[3]);
                    dropout4(drop, e0 + 4, v[4], v[5], v[6], v[7]);
                  }
                }
                const int chunk = half * 4 + j;
                st_shared_v4(srow + (uint32_t(chunk ^ sw) << 4), pack2<kODT>(v[0], v[1]),
                             pack2<kODT>(v[2], v[3]), pack2<kODT>(v[4], v[5]), pack2<kODT>(v[6], v[7]));
              }
            }
          } else if constexpr (kOut8) {
            // ---- BIAS_GELU_E4M3 (fp8 FeedForward Dense_0): e4m3(gelu(acc * wscale + bias)); the slab is 128 rows of 64 B
            // (64 columns) through a TMA map with a 64-byte box and the 64-byte swizzle: 16-byte chunk bits [4,6) of the
            // linear offset row * 64 + byte ^= its bits [7,9) ----
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t r[32];
              tmem_ld_32x32b_x32(t_row + uint32_t(s * SLAB_COLS + half * 32), r);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 2; ++j) {            // 16 columns -> one 16-byte chunk of codes
                uint32_t q[4];
#pragma unroll
                for (int h = 0; h < 2; ++h) {          // 8 columns at a time (register pressure)
                  const int nb = n0 + half * 32 + j * 16 + h * 8;   // N % 16 == 0: a chunk is wholly in or out
                  float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0, b0 = w0, b1 = w0;
                  if (nb < N) {
                    w0 = __ldg(reinterpret_cast<const float4*>(wscale + nb));
                    w1 = __ldg(reinterpret_cast<const float4*>(wscale + nb + 4));
                    b0 = __ldg(reinterpret_cast<const float4*>(bias + nb));
                    b1 = __ldg(reinterpret_cast<const float4*>(bias + nb + 4));
                  }
                  const float ws[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
                  const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                  float v[8];
#pragma unroll
                  for (int e = 0; e < 8; e += 2) {
                    const int c = j * 16 + h * 8 + e;
                    const unsigned long long y2 = fma_f32x2(pack_f32x2(__uint_as_float(r[c]), __uint_as_float(r[c + 1])),
                                                            pack_f32x2(ws[e], ws[e + 1]), pack_f32x2(bb[e], bb[e + 1]));
                    unpack_f32x2(gelu_tanh_fast2(y2), v[e], v[e + 1]);
                  }
                  q[h * 2] = pack4_e4m3(v[0], v[1], v[2], v[3]);
                  q[h * 2 + 1] = pack4_e4m3(v[4], v[5], v[6], v[7]);
                }
                const uint32_t lin = uint32_t(lrow) * 64u + uint32_t(half * 2 + j) * 16u;
                st_shared_v4(slab + (lin ^ (((lin >> 7) & 3u) << 4)), q[0], q[1], q[2], q[3]);
              }
            }
          } else {
            uint32_t r[32];
            tmem_ld_32x32b_x32(t_row + uint32_t(s * SLAB_COLS), r);
            // TOKENS: output row = token row b*T + t; t = 0 is the class-token row when cls is given
            // (vit.py:151-153: concat([cls, x]) + pos_embedding), every other row a patch row
            const int tok = kTokens ? (m_row0 + lrow) % tpi : 0;
            const bool cls_row = kTokens && cls != nullptr && tok == 0;
            const float* pos_row = aux + int64_t(tok) * N;
            uint16_t* x16_row = kLnOut ? static_cast<uint16_t*>(ln.x16) + int64_t(m_row0 + lrow) * N : nullptr;
            const bool row_ok = m_row0 + lrow < M;
            uint32_t hx[8];                            // 16-bit pairs of up to four 4-column chunks: 16 values = one 32-byte store
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 8; ++j) {              // 4 fp32 columns -> one 16-byte chunk
              const int nb = n0 + j * 4;
              float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
              if (nb < N && sp == 0 && bias != nullptr) b4 = __ldg(reinterpret_cast<const float4*>((cls_row ? cls : bias) + nb));
              float o0 = __uint_as_float(r[j * 4 + 0]), o1 = __uint_as_float(r[j * 4 + 1]);
              float o2 = __uint_as_float(r[j * 4 + 2]), o3 = __uint_as_float(r[j * 4 + 3]);
              if constexpr (kF8) {   // acc * the weight's column scale, then the bias below
                if (nb < N) {
                  const float4 w4 = __ldg(reinterpret_cast<const float4*>(wscale + nb));
                  o0 *= w4.x; o1 *= w4.y; o2 *= w4.z; o3 *= w4.w;
                }
              }
              if constexpr (kTokens) {
                if (cls_row) o0 = o1 = o2 = o3 = 0.f;   // the slot row of the patch matrix holds no data
                if (nb < N) {
                  const float4 p4 = __ldg(reinterpret_cast<const float4*>(pos_row + nb));
                  b4.x += p4.x; b4.y += p4.y; b4.z += p4.z; b4.w += p4.w;
                }
              }
              o0 += b4.x; o1 += b4.y; o2 += b4.z; o3 += b4.w;
              if constexpr (kDrop && kTokens)      // emb dropout (vit.py:155)
                dropout4(drop, int64_t(m_row0 + lrow) * N + nb, o0, o1, o2, o3);
              if constexpr (kDrop && kEpi == VITB200_EPI_BIAS_RESID_F32)   // Dropout after to_out / FF Dense_1
                dropout4(drop, int64_t(m_row0 + lrow) * N + nb, o0, o1, o2, o3);   // (vit.py:52,83), before the residual add
              if constexpr (kLoadX) {               // the Residual add (vit.py:39) happens here, on the slab TMA brought in
                const float4 xo = ld_shared_v4f(srow + (uint32_t(j ^ sw) << 4));
                o0 += xo.x; o1 += xo.y; o2 += xo.z; o3 += xo.w;
              }
              st_shared_v4(srow + (uint32_t(j ^ sw) << 4), __float_as_uint(o0), __float_as_uint(o1),
                           __float_as_uint(o2), __float_as_uint(o3));
              if constexpr (kLnOut) {
                // what the next LayerNorm needs: the row's sum and sum of squares (fp32 values, columns >= N are zero) and
                // the 16-bit copy of the raw row, the A operand of the GEMM that follows it
                st1 += (o0 + o1) + (o2 + o3);
                st2 = fmaf(o0, o0, fmaf(o1, o1, fmaf(o2, o2, fmaf(o3, o3, st2))));
                hx[(j & 3) * 2] = pack2<kDT>(o0, o1);
                hx[(j & 3) * 2 + 1] = pack2<kDT>(o2, o3);
                // every lane writes its own row, so a warp-wide store touches 32 lines whatever its width: 32-byte stores
                // (STG.256) are half the requests of 16-byte ones; N is a multiple of 8, so a row can end on a 16-byte piece
                if ((j & 3) == 3 && row_ok) {
                  if (nb + 4 <= N && (N & 15) == 0)          // rows of N 16-bit values start 32-byte aligned
                    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(x16_row + nb - 12), "r"(hx[0]), "r"(hx[1]),
                                 "r"(hx[2]), "r"(hx[3]), "r"(hx[4]), "r"(hx[5]), "r"(hx[6]), "r"(hx[7]) : "memory");
                  else {
                    if (nb - 4 <= N) *reinterpret_cast<uint4*>(x16_row + nb - 12) = make_uint4(hx[0], hx[1], hx[2], hx[3]);
                    if (nb + 4 <= N) *reinterpret_cast<uint4*>(x16_row + nb - 4) = make_uint4(hx[4], hx[5], hx[6], hx[7]);
                  }
                }
              }
            }
          }
          fence_proxy_async_smem();                    // generic-proxy smem writes -> async proxy
          named_bar_sync(1 + grp, 128);
          if (leader && !(dbg & 2)) {
            if constexpr (kEpi == VITB200_EPI_BIAS_RESID_F32)
              tma_reduce_add_2d(&tmC, slab, n0, m_row0);          // x += acc + bias
            else
              tma_store_2d(&tmC, slab, n0, m_row0);
            if constexpr (kDual) tma_store_2d(&tmC, sSlab + uint32_t(grp * 2 + (buf ^ 1)) * SLAB_BYTES, n0, m_row0 + tpi);
            tma_store_commit();
          }
          if constexpr (kLoadX) {
            // the buffer of the PREVIOUS slab is free once its store has been read out: refill it with the slab two ahead
            if (leader) { tma_store_wait_read<1>(); issue_x_load(); }
            ++x_used;
          }
          buf ^= 1;
        }
        if constexpr (kLnOut) {
          if (m_row0 + lrow < M && sp == 0)
            ln.stats[int64_t(m_row0 + lrow) * ln.slots + n_blk * 2 + grp] = make_float2(st1, st2);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CL != 1) mbar_arrive_cluster(tempty_bar(acc), lead);   // the pair leader's barrier
        else mbar_arrive(tempty_bar(acc));
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
    if (!kDirect && leader) tma_store_wait<0>();       // smem must outlive the last bulk stores
  }

  tc_fence_before();
  if constexpr (CL != 1) cluster_sync_all(); else __syncthreads();   // peer smem/TMEM stay live until here
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<MMA_CG>(tmem_base, TMEM_COLS);
  }
}

int gemm_dbg() {   // VITB200_GEMM_DBG bit 0: no TMA loads, bit 1: no output stores, bit 2: no epilogue at all
  static int v = -1;
  if (v < 0) { const char* e = getenv("VITB200_GEMM_DBG"); v = e ? atoi(e) : 0; }
  return v;
}

template <int kEpi, int kDT, int kCG, bool kDrop, bool kMN = false>
int launch_cg(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
              const CUtensorMap& tmC, const float* bias, void* C, int M, int N, int K,
              const float* aux, int tpi, const Dropout& drop, int cls_off, const float* cls, const LnFold& ln = LnFold(),
              const float* wscale = nullptr) {
  static PerDevice<bool> configured_on;   // the smem opt-in is per (function, device)
  static PerDevice<int> max_units_on;   // clusters (CTAs for kCG == 1) that can be resident at once, per device
  int& max_units = max_units_on.here();
  if (bool& configured = configured_on.here(); !configured) {
    VB_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<kEpi, kDT, kCG, kDrop, kMN>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes<kCG, kEpi>()));
    max_units = sm_count() / Cfg<kCG>::CL;
    if (Cfg<kCG>::CL > 2) {   // clusters of 4 do not tile every GPC: ask how many fit (33 on a 148-SM B200)
      int n = 0;
      cudaLaunchConfig_t cfg{};
      cfg.blockDim = dim3(NUM_THREADS);
      cfg.dynamicSmemBytes = smem_bytes<kCG, kEpi>();
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = Cfg<kCG>::CL;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      cfg.gridDim = dim3(sm_count() / Cfg<kCG>::CL * Cfg<kCG>::CL);
      if (cudaOccupancyMaxActiveClusters(&n, gemm_tc_kernel<kEpi, kDT, kCG, kDrop, kMN>, &cfg) == cudaSuccess && n > 0)
        max_units = n < max_units ? n : max_units;
      else
        cudaGetLastError();
    }
    configured = true;
  }
  const int splits = (kEpi == VITB200_EPI_BIAS_RESID_F32 && tpi > 1) ? tpi : 1;
  const int tiles = ceil_div(ceil_div(M, Cfg<kCG>::TILE_M), Cfg<kCG>::PAIRS) * ceil_div(N, Cfg<kCG>::BN_) * splits;
  const int units = tiles < max_units ? tiles : max_units;
  VB_CUDA(launch_kernel(gemm_tc_kernel<kEpi, kDT, kCG, kDrop, kMN>, dim3(units * Cfg<kCG>::CL), dim3(NUM_THREADS), smem_bytes<kCG, kEpi>(),
                        stream, Cfg<kCG>::CL, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, gemm_dbg(), drop, cls_off, cls, ln, wscale));
  VB_LAUNCH_CHECK("gemm_tc_kernel");
  return 0;
}

// the LayerNorm-fold epilogues: tile modes 1, 2 and 64, no dropout variants (the forward keeps the stand-alone
// LayerNorm kernel when a dropout rate is > 0)
template <int kEpi, int kDT>
int launch_ln(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
              const CUtensorMap& tmC, const float* bias, void* C, int M, int N, int K,
              const float* aux, int tpi, int cta_group, int cls_off, const float* cls, const LnFold& ln) {
  if (cta_group == 64) return launch_cg<kEpi, kDT, 64, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, Dropout(), cls_off, cls, ln);
  if (cta_group == 1) return launch_cg<kEpi, kDT, 1, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, Dropout(), cls_off, cls, ln);
  if (cta_group == 2) return launch_cg<kEpi, kDT, 2, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, Dropout(), cls_off, cls, ln);
  return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc: the LayerNorm-fold epilogues are built for tile modes 1, 2 and 64");
}

template <int kEpi, int kDT>
int launch_one(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
               const CUtensorMap& tmC, const float* bias, void* C, int M, int N, int K,
               const float* aux, int tpi, int cta_group, const Dropout& drop, int cls_off, const float* cls) {
  // dropout variants exist for the epilogues that have a Dropout behind them and for the two
  // production tile modes; the opt-in cluster-of-4 mode falls back to pairs when dropout is on
  constexpr bool kCanDrop = kEpi == VITB200_EPI_BIAS_GELU_16 || kEpi == VITB200_EPI_BIAS_RESID_F32 || kEpi == VITB200_EPI_BIAS_PRE_GELU_16 ||
                            kEpi == VITB200_EPI_PATCH_F32 || kEpi == VITB200_EPI_TOKENS_F32;
  if constexpr (kCanDrop) {
    if (drop.threshold != 0) {
      if (cta_group == 4)
        return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc: dropout is not built for the opt-in cluster-of-4 mode");
      if (cta_group == 64) return launch_cg<kEpi, kDT, 64, true>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
      if (cta_group == 1) return launch_cg<kEpi, kDT, 1, true>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
      return launch_cg<kEpi, kDT, 2, true>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
    }
  }
  if (cta_group == 64) return launch_cg<kEpi, kDT, 64, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
  if (cta_group == 4) return launch_cg<kEpi, kDT, 4, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
  if (cta_group == 2) return launch_cg<kEpi, kDT, 2, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
  return launch_cg<kEpi, kDT, 1, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, drop, cls_off, cls);
}

template <int kDT>
int dispatch_epi(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
                 const CUtensorMap& tmC, const float* bias, void* C, int M, int N, int K,
                 int epilogue, const float* aux, int tpi, int cta_group, const Dropout& drop, int cls_off,
                 const float* cls, const LnFold& ln) {
  if (epilogue >= VITB200_EPI_RESID_LN && epilogue <= VITB200_EPI_LN_GELU_16) {
    if (drop.threshold != 0) return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc: the LayerNorm-fold epilogues have no dropout variant");
    if (ln.stats == nullptr || ln.slots <= 0) return fail(VITB200_ERR_INVALID, "gemm_tc: LayerNorm-fold epilogue without a statistics buffer");
    const bool producer = epilogue == VITB200_EPI_RESID_LN || epilogue == VITB200_EPI_TOKENS_LN;
    if (producer && (ln.x16 == nullptr || ln.slots != 2 * ceil_div(N, cta_group == 64 ? 64 : GEMM_BN)))
      return fail(VITB200_ERR_INVALID, "gemm_tc: RESID_LN / TOKENS_LN need x16 and 2 * n_tiles statistics slots");
    if (!producer && ln.c == nullptr) return fail(VITB200_ERR_INVALID, "gemm_tc: LN_STORE / LN_GELU need the column sums c");
    switch (epilogue) {
      case VITB200_EPI_RESID_LN:
        return launch_ln<VITB200_EPI_RESID_LN, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, 0, cta_group, cls_off, cls, ln);
      case VITB200_EPI_TOKENS_LN:
        if (aux == nullptr || tpi <= 0) return fail(VITB200_ERR_INVALID, "gemm_tc: TOKENS_LN needs pos_embedding and tokens per image");
        return launch_ln<VITB200_EPI_TOKENS_LN, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, cls_off, cls, ln);
      case VITB200_EPI_LN_STORE_16:
        return launch_ln<VITB200_EPI_LN_STORE_16, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, 0, cta_group, cls_off, cls, ln);
      default:
        return launch_ln<VITB200_EPI_LN_GELU_16, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, 0, cta_group, cls_off, cls, ln);
    }
  }
  switch (epilogue) {
    case VITB200_EPI_STORE_16:
      return launch_one<VITB200_EPI_STORE_16, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_BIAS_GELU_16:
      return launch_one<VITB200_EPI_BIAS_GELU_16, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_BIAS_RESID_F32:
      return launch_one<VITB200_EPI_BIAS_RESID_F32, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_BIAS_F32:
      return launch_one<VITB200_EPI_BIAS_F32, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_PATCH_F32:
      if (aux == nullptr || tpi <= 0)
        return fail(VITB200_ERR_INVALID, "gemm_tc: PATCH epilogue needs pos_embedding and tokens");
      return launch_one<VITB200_EPI_PATCH_F32, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_BIAS_16:
      return launch_one<VITB200_EPI_BIAS_16, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_BIAS_PRE_GELU_16:
      if (tpi < M) return fail(VITB200_ERR_INVALID, "gemm_tc: PRE_GELU epilogue needs the row offset of its second output (>= M)");
      return launch_one<VITB200_EPI_BIAS_PRE_GELU_16, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    case VITB200_EPI_TOKENS_F32:
      if (aux == nullptr || tpi <= 0)
        return fail(VITB200_ERR_INVALID, "gemm_tc: TOKENS epilogue needs pos_embedding and tokens per image");
      return launch_one<VITB200_EPI_TOKENS_F32, kDT>(stream, tmA, tmB, tmC, bias, C, M, N, K, aux, tpi, cta_group, drop, cls_off, cls);
    default:
      return fail(VITB200_ERR_INVALID, "gemm_tc: unknown epilogue");
  }
}

// the fp8 GEMMs (E4M3 operands): the four epilogues of the fp8 forward, tile modes 1, 2 and 64, no dropout, no split-K
template <int kEpi>
int launch_e4m3(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                const float* bias, void* C, int M, int N, int K, int cta_group, const float* wscale) {
  if (cta_group == 64)
    return launch_cg<kEpi, DT_E4M3, 64, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, nullptr, 0, Dropout(), 1, nullptr, LnFold(), wscale);
  if (cta_group == 1)
    return launch_cg<kEpi, DT_E4M3, 1, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, nullptr, 0, Dropout(), 1, nullptr, LnFold(), wscale);
  if (cta_group == 2)
    return launch_cg<kEpi, DT_E4M3, 2, false>(stream, tmA, tmB, tmC, bias, C, M, N, K, nullptr, 0, Dropout(), 1, nullptr, LnFold(), wscale);
  return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc: E4M3 operands are built for tile modes 1, 2 and 64");
}

int dispatch_e4m3(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                  const float* bias, void* C, int M, int N, int K, int epilogue, int cta_group, const Dropout& drop,
                  const float* wscale) {
  if (wscale == nullptr) return fail(VITB200_ERR_INVALID, "gemm_tc: E4M3 operands need the per-column weight scales");
  if (drop.threshold != 0) return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc: E4M3 operands have no dropout variant");
  if ((K % 16) != 0) return fail(VITB200_ERR_INVALID, "gemm_tc: E4M3 operands need K % 16 == 0 (16-byte row pitch)");
  switch (epilogue) {
    case VITB200_EPI_STORE_16:
      return launch_e4m3<VITB200_EPI_STORE_16>(stream, tmA, tmB, tmC, bias, C, M, N, K, cta_group, wscale);
    case VITB200_EPI_BIAS_GELU_E4M3:
      if ((N % 16) != 0) return fail(VITB200_ERR_INVALID, "gemm_tc: BIAS_GELU_E4M3 needs N % 16 == 0");
      return launch_e4m3<VITB200_EPI_BIAS_GELU_E4M3>(stream, tmA, tmB, tmC, bias, C, M, N, K, cta_group, wscale);
    case VITB200_EPI_BIAS_RESID_F32:
      return launch_e4m3<VITB200_EPI_BIAS_RESID_F32>(stream, tmA, tmB, tmC, bias, C, M, N, K, cta_group, wscale);
    case VITB200_EPI_BIAS_F32:
      return launch_e4m3<VITB200_EPI_BIAS_F32>(stream, tmA, tmB, tmC, bias, C, M, N, K, cta_group, wscale);
    default:
      return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc: E4M3 operands take the STORE_16, BIAS_GELU_E4M3, BIAS_RESID_F32 and "
                                           "BIAS_F32 epilogues");
  }
}

}  // namespace

int gemm_tc_cta_group(int M) { return gemm_tc_tile_mode(M, 1 << 20); }

// Tile mode for an [M, N] output.  VITB200_GEMM_CTA_GROUP=1|2|4|64 overrides (A/B tests).  Measured
// (profiles/r01_gemm.md): CTA pairs (256x256) win from M = 1576 rows up on every ViT shape; at one or
// two row blocks (a forward at batch 1) the 128x64 single-CTA tiles are 15-25 % faster because they
// spread the weight matrix over four times as many SMs, and lose badly beyond that (their MMAs run
// at a quarter of the rate).  The weight-multicast cluster of two pairs (4) is no faster per SM and
// fits only 33 clusters on 148 SMs (DESIGN.md): opt-in only.
int gemm_tc_tile_mode(int M, int N) {
  // read on every call (a getenv per GEMM launch is noise): the per-kernel tests switch modes in-process
  const char* e = getenv("VITB200_GEMM_CTA_GROUP");
  const int forced = e ? atoi(e) : 0;
  if (forced == 1 || forced == 2 || forced == 4 || forced == 64) return forced;
  if (M <= 2 * GEMM_BM) return N > GEMM_BN ? 64 : 1;
  return 2;
}

int launch_gemm_tc_wgrad(cudaStream_t stream, const CUtensorMap& tmX, const CUtensorMap& tmdY, const CUtensorMap& tmC,
                         const float* zero_bias, float* C, int M, int N, int K, int splits, int dtype, int cta_group) {   // zero_bias may be null
  if (M <= 0 || N <= 0 || K <= 0) return fail(VITB200_ERR_INVALID, "gemm_tc_wgrad: empty problem");
  if ((M % 8) != 0 || (N % 8) != 0) return fail(VITB200_ERR_INVALID, "gemm_tc_wgrad: M and N must be multiples of 8");
  const int num_kb = ceil_div(K, GEMM_BK);
  int sp = splits < 1 ? 1 : (splits > num_kb ? num_kb : splits);
  sp = ceil_div(num_kb, ceil_div(num_kb, sp));
  constexpr int E = VITB200_EPI_BIAS_RESID_F32;
#define VB_WGRAD(DT)                                                                                                     \
  do {                                                                                                                   \
    if (cta_group == 64) return launch_cg<E, DT, 64, false, true>(stream, tmX, tmdY, tmC, zero_bias, C, M, N, K, nullptr, sp, Dropout(), 1, nullptr); \
    if (cta_group == 1) return launch_cg<E, DT, 1, false, true>(stream, tmX, tmdY, tmC, zero_bias, C, M, N, K, nullptr, sp, Dropout(), 1, nullptr);   \
    return launch_cg<E, DT, 2, false, true>(stream, tmX, tmdY, tmC, zero_bias, C, M, N, K, nullptr, sp, Dropout(), 1, nullptr);                        \
  } while (0)
  if (dtype == DT_BF16) VB_WGRAD(DT_BF16);
  if (dtype == DT_F16) VB_WGRAD(DT_F16);
#undef VB_WGRAD
  return fail(VITB200_ERR_INVALID, "gemm_tc_wgrad: dtype must be bf16 or fp16");
}

int launch_gemm_tc(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
                   const CUtensorMap* tmC, const float* bias, void* C, int M, int N, int K,
                   int epilogue, const float* aux, int tpi, int dtype, int cta_group, const Dropout& drop,
                   int cls_off, const float* cls, const LnFold& ln, const float* wscale) {
  if (cta_group != 1 && cta_group != 2 && cta_group != 4 && cta_group != 64)
    return fail(VITB200_ERR_INVALID, "gemm_tc: tile mode must be 1, 2, 4 or 64");
  if (M <= 0 || N <= 0 || K <= 0) return fail(VITB200_ERR_INVALID, "gemm_tc: empty problem");
  if ((N % 8) != 0 || (K % 8) != 0)
    return fail(VITB200_ERR_INVALID, "gemm_tc: N and K must be multiples of 8");
  if (epilogue != VITB200_EPI_STORE_16 && bias == nullptr)
    return fail(VITB200_ERR_INVALID, "gemm_tc: epilogue needs a bias");
  if (epilogue != VITB200_EPI_PATCH_F32 && tmC == nullptr)
    return fail(VITB200_ERR_INVALID, "gemm_tc: output tensor map missing");
  if (dtype == DT_E4M3) {
    if (tmC == nullptr) return fail(VITB200_ERR_INVALID, "gemm_tc: output tensor map missing");
    if (epilogue != VITB200_EPI_STORE_16 && bias == nullptr) return fail(VITB200_ERR_INVALID, "gemm_tc: epilogue needs a bias");
    return dispatch_e4m3(stream, tmA, tmB, *tmC, bias, C, M, N, K, epilogue, cta_group, drop, wscale);
  }
  if (epilogue == VITB200_EPI_BIAS_RESID_F32) {
    // `tpi` = split-K factor: clamp so that every split owns at least one k-block
    const int num_kb = ceil_div(K, GEMM_BK);
    int sp = tpi < 1 ? 1 : (tpi > num_kb ? num_kb : tpi);
    sp = ceil_div(num_kb, ceil_div(num_kb, sp));
    tpi = sp;
  }
  const CUtensorMap& c = tmC ? *tmC : tmA;   // PATCH never touches it
  const float* cls_p = (cls_off == 1 && (epilogue == VITB200_EPI_PATCH_F32 || epilogue == VITB200_EPI_TOKENS_F32 ||
                                         epilogue == VITB200_EPI_TOKENS_LN)) ? cls : nullptr;
  if (dtype == DT_BF16)
    return dispatch_epi<DT_BF16>(stream, tmA, tmB, c, bias, C, M, N, K, epilogue, aux, tpi, cta_group, drop, cls_off, cls_p, ln);
  if (dtype == DT_F16)
    return dispatch_epi<DT_F16>(stream, tmA, tmB, c, bias, C, M, N, K, epilogue, aux, tpi, cta_group, drop, cls_off, cls_p, ln);
  return fail(VITB200_ERR_INVALID, "gemm_tc: dtype must be bf16, fp16 or E4M3");
}

}  // namespace vb
