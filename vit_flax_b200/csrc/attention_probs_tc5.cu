// attention_probs_tc5.cu -- the attention weights of one layer, P = softmax(Q K^T * 64^-0.5) (vit.py:73-75), as fp32
// [B, h, T, T] rows of a caller's tensor: what vit-pytorch's Recorder returns and attention maps / rollout start from.
//
// The fused attention kernels never materialise P (it lives in TMEM as unnormalised 16-bit pairs and TMEM and shared
// memory are full: DESIGN.md section 3 K4), so P is RECOMPUTED next to the forward from the same 16-bit q / k and the
// row log-sum-exp the forward kernel writes when asked (its `lse` argument, the identity of attention_bwd_tc5.cu):
//
//   P_ij = exp2(s_ij * sl2 - lse2_i)     s = Q K^T,  sl2 = 64^-0.5 * log2(e),  lse2_i = log2 sum_j exp2(s_ij sl2)
//
// No row maximum and no second pass: every (query tile, key block) is independent.
// One work item = (image, head, 128-query tile); persistent CTAs take contiguous ranges of items, so the q tiles of an
// (image, head) run back to back and re-read its K blocks from L2.  A CTA walks the FLAT sequence of (item, key block)
// pairs, so the pipelines run across item boundaries.  12 warps:
//   warp 0  lane 0 : TMA producer -- the Q tile and the K blocks of 128 keys cut out of the to_qkv output [B, T, 3I]
//                    (the boxes and coordinates of the forward kernels); rows >= T arrive as zeros.  Q: 2-deep ring
//                    (one tile per item), K: 4-deep ring (one block per step).
//   warp 1  lane 0 : tcgen05.mma issuer: S = Q K_j^T (M = 128, N = 128, K = 64, kind::f16, SS operands) into one of two
//                    TMEM slots of 128 fp32 columns, so block j+1 is computed while block j is drained.
//   warp 2         : TMEM allocator (256 columns).
//   warps 4..11    : math, thread = query row = TMEM lane; the two warps of a lane quarter take 64 key columns each.  A
//                    warp pulls its columns out of TMEM (the slot is released at once), exponentiates, and writes
//                    32 x 32 tiles through a private shared-memory transpose: a row of the output is 4 T bytes long, not
//                    a 16-byte multiple at T = 197 or 257, so no TMA tensor store; instead every warp-wide store covers
//                    32 consecutive floats of ONE row (coalesced, streaming .cs).  Only elements inside [T, T] are written.
// Bound: the writes -- 4 T^2 bytes per (image, head); the recompute is 2 T^2 64 flops on the tensor cores.
#include "common.h"
#include "ptx.cuh"

namespace vb {

namespace {

constexpr int DH = 64;
constexpr int QT = 128;                  // queries per item (UMMA M)
constexpr int KB = 128;                  // keys per block (UMMA N)
constexpr int NT = 384;                  // 4 service warps + 8 math warps
constexpr int TILE_BYTES = 128 * 128;    // 128 rows x 64 16-bit features (128-byte swizzle)
constexpr int QS = 2, KS = 4;            // Q / K ring depths
constexpr int STG_LD = 36;               // staging row pitch in floats (16-byte aligned rows; 4-way bank split per v4 store)
constexpr int STG_FLOATS = 32 * STG_LD;  // one 32 x 32 tile per math warp
constexpr int OFF_Q = 0;
constexpr int OFF_K = OFF_Q + QS * TILE_BYTES;
constexpr int OFF_STG = OFF_K + KS * TILE_BYTES;
constexpr int OFF_BAR = OFF_STG + 8 * STG_FLOATS * 4;
constexpr int SMEM_TOTAL = OFF_BAR + 256 + 1024 /*align slack*/;
constexpr uint32_t TMEM_COLS = 2 * KB;
static_assert(SMEM_TOTAL <= 232448, "shared memory budget");

template <int kDT>
__global__ void __launch_bounds__(NT, 1)
attention_probs_tc5_kernel(const __grid_constant__ CUtensorMap tmQKV,   // qkv [B, T, 3I], box 128 rows x 64
                           const float* __restrict__ lse2, float* __restrict__ out, int64_t img_stride,
                           int T, int heads, int nqt, int nkb, int items) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQ = base + OFF_Q, sK = base + OFF_K, bars = base + OFF_BAR;
  auto q_full = [&](int s) { return bars + 8u * (0 + s); };     // [QS]
  auto q_empty = [&](int s) { return bars + 8u * (2 + s); };
  auto k_full = [&](int s) { return bars + 8u * (4 + s); };     // [KS]
  auto k_empty = [&](int s) { return bars + 8u * (8 + s); };
  auto s_full = [&](int s) { return bars + 8u * (12 + s); };    // [2 TMEM slots]
  auto s_empty = [&](int s) { return bars + 8u * (14 + s); };
  const uint32_t tmem_slot = bars + 8u * 16;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + OFF_BAR + 8 * 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = heads * DH;
  const int64_t first = int64_t(blockIdx.x) * items / gridDim.x;
  const int64_t last = int64_t(blockIdx.x + 1) * items / gridDim.x;
  const int G = int(last - first) * nkb;                         // (item, key block) steps of this CTA

  if (warp == 0 && lane == 0) prefetch_tmap(&tmQKV);
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < QS; ++s) { mbar_init(q_full(s), 1); mbar_init(q_empty(s), 1); }
    for (int s = 0; s < KS; ++s) { mbar_init(k_full(s), 1); mbar_init(k_empty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(s_full(s), 1); mbar_init(s_empty(s), 8); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<1>(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_launch_dependents();
  pdl_wait();                // the attention kernel (and with it the to_qkv GEMM) has completed: q, k and lse2 are final

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      for (int g = 0; g < G; ++g) {
        const int i = g / nkb, kb = g - i * nkb;
        const int64_t item = first + i;
        const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
        const int b = bh / heads, h = bh - b * heads;
        if (kb == 0) {
          const int qs = i & (QS - 1);
          mbar_wait(q_empty(qs), ((i / QS) & 1) ^ 1u);
          mbar_arrive_expect_tx(q_full(qs), TILE_BYTES);
          tma_load_3d(sQ + qs * TILE_BYTES, &tmQKV, q_full(qs), h * DH, qt * QT, b);
        }
        const int ks = g & (KS - 1);
        mbar_wait(k_empty(ks), ((g / KS) & 1) ^ 1u);
        mbar_arrive_expect_tx(k_full(ks), TILE_BYTES);
        tma_load_3d(sK + ks * TILE_BYTES, &tmQKV, k_full(ks), inner + h * DH, kb * KB, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_16(QT, KB, kDT == DT_F16 ? 0 : 1, 0);   // both operands K-major
      for (int g = 0; g < G; ++g) {
        const int i = g / nkb, kb = g - i * nkb;
        const int qs = i & (QS - 1), ks = g & (KS - 1), s = g & 1;
        if (kb == 0) mbar_wait(q_full(qs), (i / QS) & 1);
        mbar_wait(k_full(ks), (g / KS) & 1);
        mbar_wait(s_empty(s), ((g >> 1) & 1) ^ 1u);               // the math warps have read this slot's last block
        tc_fence_after();
        const uint32_t q0 = sQ + qs * TILE_BYTES, k0 = sK + ks * TILE_BYTES;
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)                         // 16 features = 32 B along the swizzled row
          umma_bf16_ss<1>(tmem_base + uint32_t(s) * KB, umma_desc_k_sw128(q0 + k * 32), umma_desc_k_sw128(k0 + k * 32),
                          idesc, k != 0 ? 1u : 0u);
        umma_commit(k_empty(ks));
        if (kb == nkb - 1) umma_commit(q_empty(qs));
        umma_commit(s_full(s));
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== math: thread = query row, two warps per lane quarter split the block's keys =====================
    const int w = warp - 4, q = w & 3, half = w >> 2;          // q == warp % 4: the TMEM lane quarter this warp may read
    const uint32_t t_lane = tmem_base + (uint32_t(q * 32) << 16);
    const float sl2 = 0.125f * 1.4426950408889634f;          // dim_head^-0.5 * log2(e)   (vit.py:66)
    float* stg = reinterpret_cast<float*>(gbase + OFF_STG) + w * STG_FLOATS;
    const uint32_t stg_u32 = smem_u32(stg);
    float lse = 0.f;
    for (int g = 0; g < G; ++g) {
      const int i = g / nkb, kb = g - i * nkb;
      const int64_t item = first + i;
      const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
      const int b = bh / heads, h = bh - b * heads;
      const int q0 = qt * QT + q * 32;                          // first query row of this warp
      const int rows = min(32, T - q0);                         // valid rows of the warp (<= 0: none)
      const int c0 = kb * KB + half * 64;                       // first key column of this warp
      const int nch = rows > 0 ? max(0, min(2, (T - c0 + 31) / 32)) : 0;   // 32-key chunks holding a key < T
      if (kb == 0) lse = (q0 + lane < T) ? __ldg(lse2 + (int64_t(bh) * T + q0 + lane)) : 0.f;
      const int s = g & 1;
      mbar_wait(s_full(s), (g >> 1) & 1);
      tc_fence_after();
      uint32_t v[64];
      if (nch > 0) {
        tmem_ld_32x32b_x32p(t_lane + uint32_t(s * KB + half * 64), v);
        if (nch > 1) tmem_ld_32x32b_x32p(t_lane + uint32_t(s * KB + half * 64 + 32), v + 32);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty(s));                   // the scores are in registers: the next block may land
      float* dst_row0 = out + int64_t(b) * img_stride + (int64_t(h) * T + q0) * T;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        if (c < nch) {
          // this row's 32 probabilities -> row `lane` of the staging tile
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float p[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {   // <= 1 like every softmax value: a row ruled by one key gets exp2 of the
                                            // fp32 rounding of lse2 (m sl2 of a large maximum), a few 1e-6 above 1.
                                            // Not fminf: a NaN score (non-finite q / k) must stay NaN, not become 1
              const float pe = ex2_approx(fmaf(__uint_as_float(v[c * 32 + j + e]), sl2, -lse));
              p[e] = pe > 1.0f ? 1.0f : pe;
            }
            st_shared_v4(stg_u32 + uint32_t(lane * STG_LD + j) * 4u, __float_as_uint(p[0]), __float_as_uint(p[1]),
                         __float_as_uint(p[2]), __float_as_uint(p[3]));
          }
          __syncwarp();
          // column `lane` of the tile, row by row: each store is 32 consecutive floats of one output row
          const int col = c0 + c * 32 + lane;
          if (col < T) {
            float* dst = dst_row0 + col;
#pragma unroll 8
            for (int rr = 0; rr < 32; ++rr)
              if (rr < rows) __stcs(dst + int64_t(rr) * T, stg[rr * STG_LD + lane]);
          }
          __syncwarp();                                         // the tile is read out before the next chunk overwrites it
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, TMEM_COLS);
  }
}

template <int kDT>
int launch_t(cudaStream_t st, const void* qkv, const float* lse2, float* out, int64_t img_stride, int batch, int T,
             int heads) {
  static PerDevice<bool> configured_on;   // the smem opt-in is per (function, device)
  if (bool& configured = configured_on.here(); !configured) {
    VB_CUDA(cudaFuncSetAttribute(attention_probs_tc5_kernel<kDT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL));
    configured = true;
  }
  const int inner = heads * DH;
  CUtensorMap tm;
  int rc;
  if ((rc = make_tmap_3d_16(&tm, qkv, batch, T, 3 * inner, 3 * inner, QT, kDT))) return rc;
  const int nqt = ceil_div(T, QT), nkb = ceil_div(T, KB);
  const int64_t items64 = int64_t(batch) * heads * nqt;
  if (items64 * nkb > 0x7fffffff) return fail(VITB200_ERR_INVALID, "attention_probs: too many work items");
  const int items = int(items64);
  const int grid = items < sm_count() ? items : sm_count();
  VB_CUDA(launch_kernel(attention_probs_tc5_kernel<kDT>, dim3(grid), dim3(NT), SMEM_TOTAL, st, 1, tm, lse2, out, img_stride,
                        T, heads, nqt, nkb, items));
  VB_LAUNCH_CHECK("attention_probs_tc5_kernel");
  return 0;
}

}  // namespace

int launch_attention_probs(cudaStream_t stream, const void* qkv, const float* lse2, float* out, int64_t img_stride,
                           int batch, int T, int heads, int dtype) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention_probs: empty problem");
  if (qkv == nullptr || lse2 == nullptr || out == nullptr) return fail(VITB200_ERR_INVALID, "attention_probs: null pointer");
  if (img_stride < int64_t(heads) * T * T) return fail(VITB200_ERR_INVALID, "attention_probs: image stride below heads * T * T");
  if (dtype == DT_BF16) return launch_t<DT_BF16>(stream, qkv, lse2, out, img_stride, batch, T, heads);
  if (dtype == DT_F16) return launch_t<DT_F16>(stream, qkv, lse2, out, img_stride, batch, T, heads);
  return fail(VITB200_ERR_INVALID, "attention_probs: dtype must be bf16 or fp16");
}

}  // namespace vb
