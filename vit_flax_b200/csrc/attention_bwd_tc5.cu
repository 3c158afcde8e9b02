// attention_bwd_tc5.cu -- attention adjoint on tcgen05 / TMEM for sequences of up to 208 tokens (every 224-px /16
// config).  Adjoint of vit.py:69-79 per (image, head):
//
//   P  = exp2(Q K^T * sl2 - lse2)            sl2 = 64^-0.5 * log2(e), lse2 = log2 sum_j exp2(s_ij sl2) from the forward
//   dV = P^T dO          dP = dO V^T          D_i = sum_d dO_id O_id   (attn_bwd_rowdot_kernel, or the statistics kernel)
//   dS = P o (dP - D) * 64^-0.5               dQ = dS K            dK = dS^T Q
//
// An (image, head) is walked in (key tile, query tile) blocks of 128 x 128 (tails 128 x 80 / 80 x 128 at T = 197), and a
// CTA works through a FLAT sequence of blocks -- its items back to back -- so every pipeline below runs across item
// boundaries.  Per block all five products are on the tensor cores:
//
//   S  = Q_q K_k^T,  dP = dO_q V_k^T   (SS, both K-major) -> TMEM fp32, computed in two 64-key halves with their own
//        barriers: the halves ARE the double buffer (a half is released as soon as it is in registers), no extra TMEM
//   thread = query row (TMEM lane): p = exp2(s sl2 - lse2), ds = p (dp - D) / 8; P and dS go to shared memory as 16-bit
//        tiles of 128 rows x 64-key atoms (128-byte swizzle).  ONE such tile serves both orientations:
//          as a K-major  A operand  [M = query, K = key]  (dQ += dS K_k)
//          as an MN-major A operand [M = key,   K = query] (dV += P^T dO_q, dK += dS^T Q_q) -- the transposes of the
//        adjoint are descriptor bits, nothing is moved.
//   dV_k += P^T dO_q,  dK_k += dS^T Q_q   accumulate over the query tiles in TMEM (64 columns each)
//   dQ_q += dS K_k                        accumulates over the key tiles in TMEM (64 columns per query tile)
//
// Two modes of the same kernel.  RESIDENT (T <= 208, kStream = false): the unit of work is an (image, head), its blocks
// run key tile outermost, and dQ of both query tiles accumulates over the key tiles in TMEM (2 x 64 columns) and leaves
// once per item.  STREAMED (any T, kStream = true): the unit is an (image, head, key tile) -- its blocks are the query
// tiles -- so dK / dV still accumulate in TMEM, while the block's dQ contribution (a fresh 64-column accumulator, two of
// them alternating) is added into an fp32 buffer [B T, heads 64] with 16-byte vector reductions (red.global.add.v4.f32)
// by the epilogue warps and converted to 16 bits by a last pass; ViT-H/14 (257 tokens) and 512-px inputs (1025) run it.
// Operands: the four 128-row tiles a block needs (Q_q, dO_q, K_k, V_k: 64 KB, TMA boxes cut out of the to_qkv output /
// the cotangent, rows past T zero-filled) stream through a two-deep ring, loaded a block ahead -- also across items.
// TMEM: S 128 + dP 128 + dV 64 + dK 64 + dQ 2 x 64 = 512 columns.  The softmax is NOT recomputed from scratch: the row
// log-sum-exp comes from the forward kernel (attention_tc5 writes it when asked), so no pass needs a row maximum and the
// blocks are independent; the MMA thread issues the next block's S / dP halves ahead of this block's dV / dK / dQ.
// Warps: 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 4..11 math (thread = query row; the two warps of a lane quarter
// split a half's key columns), 12..15 epilogue (dK / dV per key tile, dQ per item -> 16-bit rows of dqkv).
// Bound: the XU pipe -- one ex2 and two fp32->16-bit packs per score, 16 cycles per score pair per SMSP.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "common.h"
#include "ptx.cuh"

namespace vb {

#ifdef VITB200_TRACE
// debug timeline of CTA 0: g_trace_bwd[event][block] = clock64 at the event (profiles/trace_attention_bwd.py)
__device__ long long g_trace_bwd[16][64];
#define TRACEB(ev, i) do { if (blockIdx.x == 0 && (i) < 64) g_trace_bwd[ev][i] = clock64(); } while (0)
#else
#define TRACEB(ev, i) do { } while (0)
#endif

namespace {

constexpr int DH = 64;
constexpr int BT = 128;                      // block edge (UMMA M)
constexpr int NTHR = 512;
constexpr int ROWS_MAX = 208;                // longest RESIDENT sequence (dQ of at most two query tiles stays in TMEM)
constexpr int ATOM_BYTES = BT * 128;         // 128 rows x 64 columns of 16 bits: one operand tile, one 64-key atom of P / dS
constexpr int PAIR_BYTES = 2 * ATOM_BYTES;   // (K_k, V_k) or (Q_q, dO_q): two operand tiles that are loaded and released together
constexpr int OFF_KV = 0, OFF_QDO = 2 * PAIR_BYTES;   // two slots of each
constexpr int OFF_P = 4 * PAIR_BYTES, OFF_DS = OFF_P + 2 * ATOM_BYTES;
constexpr int OFF_BAR = OFF_DS + 4 * ATOM_BYTES;      // two dS tiles (consecutive blocks alternate), one P tile
constexpr int SMEM_TOTAL = OFF_BAR + 256 + 1024;
constexpr uint32_t COL_S = 0, COL_DP = 128, COL_DV = 256, COL_DK = 320, COL_DQ = 384;   // TMEM columns

template <int kDT, bool kStream>
__global__ void __launch_bounds__(NTHR, 1)
attention_bwd_tc5_kernel(const __grid_constant__ CUtensorMap tmQKV,   // qkv [B, T, 3I], box 128 rows x 64
                         const __grid_constant__ CUtensorMap tmDO,    // d_out [B, T, I], box 128 rows x 64
                         const float* __restrict__ lse2, const float* __restrict__ dsum,
                         uint16_t* __restrict__ dqkv, float* __restrict__ dq_acc, int T, int heads, int items) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sP = base + OFF_P, sDS = base + OFF_DS, bars = base + OFF_BAR;
  const uint32_t kv_full0 = bars /* [2] */, kv_empty0 = bars + 16 /* [2] */, pds_ready = bars + 32, p_free = bars + 40,
                 ds_free0 = bars + 48 /* [2] */, dkv_ready = bars + 64, dkv_free = bars + 72,
                 sdp_ready0 = bars + 96 /* [2]: per 64-key half of a block */, sdp_free0 = bars + 112 /* [2] */,
                 tmem_slot = bars + 128, dq_ready0 = bars + 144 /* [2]: resident mode uses [0] */, dq_free0 = bars + 160 /* [2] */,
                 qdo_full0 = bars + 176 /* [2] */, qdo_empty0 = bars + 192 /* [2] */;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + OFF_BAR + 128);
  // operand tiles: (K, V) pair slot s, (Q, dO) pair slot s
  auto sK = [&](int s) { return base + OFF_KV + uint32_t(s) * PAIR_BYTES; };
  auto sV = [&](int s) { return base + OFF_KV + uint32_t(s) * PAIR_BYTES + ATOM_BYTES; };
  auto sQ = [&](int s) { return base + OFF_QDO + uint32_t(s) * PAIR_BYTES; };
  auto sDO = [&](int s) { return base + OFF_QDO + uint32_t(s) * PAIR_BYTES + ATOM_BYTES; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = heads * DH;
  const int TP = (T + 15) & ~15;                             // rows the MMAs see (zero-filled past T by TMA)
  const int ntile = (T + BT - 1) / BT;                       // key tiles == query tiles (resident: 1 or 2)
  auto ext = [&](int t) { return min(BT, TP - t * BT); };    // valid (padded) rows of tile t: 128, or 80 at T = 197
  // unit of work: resident = an (image, head), ntile^2 blocks, key tile outermost; streamed = an (image, head, key tile),
  // ntile blocks (its query tiles).  A CTA takes units blockIdx.x, blockIdx.x + gridDim.x, ... and walks their blocks as
  // ONE flat sequence g -> (unit g / nb, block g % nb).
  const int nb = kStream ? ntile : ntile * ntile;
  const int units = kStream ? items * ntile : items;
  const int my_units = int(blockIdx.x) < units ? (units - 1 - int(blockIdx.x)) / int(gridDim.x) + 1 : 0;
  const int G = my_units * nb;
  // Operand pairs are loaded ONCE per use span and released after their last use.  Resident: (K, V) of key tile kt in slot
  // kt for the blocks (kt, *), (Q, dO) of query tile qt in slot qt for the blocks (*, qt) -- every tile of an item is
  // loaded once, and the next item's tiles arrive while this item's later blocks run.  Streamed: (K, V) once per unit
  // (slots alternate per unit), (Q, dO) per block (slots alternate per block).
  struct Blk { int item, kt, qt, j, kvs, qs; uint32_t kvph, qph; bool kv_first, kv_last, q_first, q_last; };
  auto block_of = [&](int g) {
    const int un = g / nb, u = int(blockIdx.x) + un * int(gridDim.x), j = g - un * nb;
    Blk b;
    b.j = j;
    if (kStream) {
      b.item = u / ntile; b.kt = u - b.item * ntile; b.qt = j;
      b.kvs = un & 1; b.kvph = uint32_t(un >> 1) & 1u; b.kv_first = j == 0; b.kv_last = j == nb - 1;
      b.qs = g & 1; b.qph = uint32_t(g >> 1) & 1u; b.q_first = true; b.q_last = true;
    } else {
      b.item = u; b.kt = j / ntile; b.qt = j - b.kt * ntile;
      b.kv_first = b.qt == 0; b.kv_last = b.qt == ntile - 1;
      b.q_first = b.kt == 0;  b.q_last = b.kt == ntile - 1;
      if (ntile == 1) {          // one block per item: the two slots alternate between items
        b.kvs = b.qs = un & 1; b.kvph = b.qph = uint32_t(un >> 1) & 1u;
      } else {
        b.kvs = b.kt; b.qs = b.qt; b.kvph = b.qph = uint32_t(un) & 1u;
      }
    }
    return b;
  };

  if (warp == 0 && lane == 0) { prefetch_tmap(&tmQKV); prefetch_tmap(&tmDO); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(kv_full0 + 8 * i, 1);    mbar_init(kv_empty0 + 8 * i, 1);
      mbar_init(qdo_full0 + 8 * i, 1);   mbar_init(qdo_empty0 + 8 * i, 1);
      mbar_init(sdp_ready0 + 8 * i, 1);  mbar_init(sdp_free0 + 8 * i, 8);
      mbar_init(ds_free0 + 8 * i, 1);
    }
    mbar_init(pds_ready, 8); mbar_init(p_free, 1);
    mbar_init(dkv_ready, 1); mbar_init(dkv_free, 4);
    for (int i = 0; i < 2; ++i) { mbar_init(dq_ready0 + 8 * i, 1); mbar_init(dq_free0 + 8 * i, 4); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<1>(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer: the four operand tiles of every block, one block ahead =====================
    if (elect_one()) {
      for (int g = 0; g < G; ++g) {
        const Blk bk = block_of(g);
        const int kt = bk.kt, qt = bk.qt;
        const int b = bk.item / heads, h = bk.item - b * heads;
        if (bk.kv_first) {
          mbar_wait(kv_empty0 + 8u * bk.kvs, bk.kvph ^ 1u);
          TRACEB(10, g);
          mbar_arrive_expect_tx(kv_full0 + 8u * bk.kvs, PAIR_BYTES);
          tma_load_3d(sK(bk.kvs), &tmQKV, kv_full0 + 8u * bk.kvs, inner + h * DH, kt * BT, b);
          tma_load_3d(sV(bk.kvs), &tmQKV, kv_full0 + 8u * bk.kvs, 2 * inner + h * DH, kt * BT, b);
        }
        if (bk.q_first) {
          mbar_wait(qdo_empty0 + 8u * bk.qs, bk.qph ^ 1u);
          mbar_arrive_expect_tx(qdo_full0 + 8u * bk.qs, PAIR_BYTES);
          tma_load_3d(sQ(bk.qs), &tmQKV, qdo_full0 + 8u * bk.qs, h * DH, qt * BT, b);
          tma_load_3d(sDO(bk.qs), &tmDO, qdo_full0 + 8u * bk.qs, h * DH, qt * BT, b);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr int fmt = kDT == DT_F16 ? 0 : 1;
      const uint32_t d_s = tmem_base + COL_S, d_dp = tmem_base + COL_DP, d_dv = tmem_base + COL_DV, d_dk = tmem_base + COL_DK;
      constexpr uint32_t idesc_t = umma_idesc_16(BT, DH, fmt, 1, 1);          // A and B MN-major: dV, dK
      constexpr uint32_t idesc_q = umma_idesc_16(BT, DH, fmt, 1, 0);          // A K-major, B MN-major: dQ
      // half hf (64 keys) of S = Q_q K_k^T and dP = dO_q V_k^T of block g, once the math warps have read the previous block's
      auto issue_half = [&](int g, int hf) {
        const Blk nx = block_of(g);
        const int kt = nx.kt;
        const uint32_t bph = uint32_t(g & 1);
        if (hf == 0) {                                                        // the block's operand pairs have arrived
          mbar_wait(kv_full0 + 8u * nx.kvs, nx.kvph);
          mbar_wait(qdo_full0 + 8u * nx.qs, nx.qph);
        }
        const int nkh = max(0, min(64, ext(kt) - 64 * hf));                   // keys of this half: 64, 16 (T = 197 tail) or 0
        mbar_wait(sdp_free0 + 8u * hf, bph ^ 1u);
        if (nkh > 0) {
          const uint32_t k_lo = umma_desc_lo(sK(nx.kvs) + hf * 8192), v_lo = umma_desc_lo(sV(nx.kvs) + hf * 8192),
                         q_lo = umma_desc_lo(sQ(nx.qs)), do_lo = umma_desc_lo(sDO(nx.qs));
          const uint32_t idesc_s = umma_idesc_16(BT, nkh, fmt, 0, 0);         // [128 q] x [nkh keys], both K-major
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < DH / 16; ++k) {                                 // 16 features = 32 B along the swizzled row
            umma_bf16_ss_lo(d_s + 64 * hf, q_lo + 2 * k, k_lo + 2 * k, idesc_s, k != 0 ? 1u : 0u);
            umma_bf16_ss_lo(d_dp + 64 * hf, do_lo + 2 * k, v_lo + 2 * k, idesc_s, k != 0 ? 1u : 0u);
          }
        }
        umma_commit(sdp_ready0 + 8u * hf);
      };
      int kti = 0;
      if (G > 0) {
        issue_half(0, 0);
        issue_half(0, 1);
      }
      for (int g = 0; g < G; ++g) {
        const Blk bk = block_of(g);
        const int it = g / nb, j = bk.j, kt = bk.kt, qt = bk.qt;
        const int nk = ext(kt), nq = ext(qt);
        const uint32_t bph = uint32_t(g & 1);
        const uint32_t ds_tile = sDS + uint32_t(g & 1) * 2 * ATOM_BYTES;
        // the next block's first half as soon as this block's has been read, its second half right after this block's math
        if (g + 1 < G) {
          TRACEB(11, g + 1);
          issue_half(g + 1, 0);
        }
        TRACEB(0, g);
        mbar_wait(pds_ready, bph);                         // P and dS of this block are in shared memory
        TRACEB(1, g);
        // Order of issue (one tcgen05.mma costs the issuing thread ~50 cycles whatever its size --
        // profiles/microbench/mma_chain.cu -- so a block's 40 are ~2 k cycles): dV first, so that the single P tile is
        // released to the next block's math warps early; then the next block's second half of S / dP; dK and dQ last (the
        // dS tile is double-buffered).  Measured against "everything after the next block's halves": the same step time
        // (24.3 ms of backward at ViT-B/16 batch 256 either way, gpurun_out/r03c_train.log) -- the P tile is not what the
        // math warps wait for.
        // ---- dV_k += P^T dO_q : A = the P tile read MN-major (M = key, K = query), B = dO_q MN-major ----
        if (qt == 0) { mbar_wait(dkv_free, uint32_t(kti & 1) ^ 1u); }         // the previous key tile's dK / dV were drained
        tc_fence_after();
        // descriptor low words: a k-step of 16 queries / keys is 2048 B further in an MN-major tile (+128), the dS tile read
        // K-major advances 32 B inside its 64-key atom (+2) and one atom (+1024) every four steps
        const uint32_t p_lo = umma_desc_lo(sP, ATOM_BYTES), ds_mn_lo = umma_desc_lo(ds_tile, ATOM_BYTES), ds_k_lo = umma_desc_lo(ds_tile),
                       do_lo = umma_desc_lo(sDO(bk.qs)), q_lo = umma_desc_lo(sQ(bk.qs)), kmn_lo = umma_desc_lo(sK(bk.kvs));
        const int nqs = nq / 16, nks = nk / 16;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          if (kk < nqs) umma_bf16_ss_lo(d_dv, p_lo + 128 * kk, do_lo + 128 * kk, idesc_t, (qt != 0 || kk != 0) ? 1u : 0u);
        umma_commit(p_free);
        TRACEB(2, g);
        if (g + 1 < G) issue_half(g + 1, 1);
        TRACEB(3, g);
        // ---- dK_k += dS^T Q_q (A = the dS tile read MN-major) and dQ_q += dS K_k (A = the dS tile read K-major, B = K_k
        //      MN-major).  dQ: resident = one accumulator per query tile, kept over the item's key tiles; streamed = a fresh
        //      accumulator per block, two alternating, drained by the epilogue warps a block later
        const uint32_t d_dq = tmem_base + COL_DQ + uint32_t(kStream ? (g & 1) : qt) * DH;
        if (kStream) mbar_wait(dq_free0 + 8u * uint32_t(g & 1), (uint32_t(g >> 1) & 1u) ^ 1u);
        else if (j == 0) mbar_wait(dq_free0, uint32_t(it & 1) ^ 1u);          // the previous item's dQ was drained
        const bool dq_fresh = kStream || kt == 0;
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          if (kk < nqs) umma_bf16_ss_lo(d_dk, ds_mn_lo + 128 * kk, q_lo + 128 * kk, idesc_t, (qt != 0 || kk != 0) ? 1u : 0u);
          if (kk < nks) umma_bf16_ss_lo(d_dq, ds_k_lo + 1024 * (kk >> 2) + 2 * (kk & 3), kmn_lo + 128 * kk, idesc_q, (!dq_fresh || kk != 0) ? 1u : 0u);
        }
        umma_commit(ds_free0 + 8u * uint32_t(g & 1));
        if (bk.kv_last) umma_commit(kv_empty0 + 8u * uint32_t(bk.kvs));    // the last block that reads this (K, V) pair
        if (bk.q_last) umma_commit(qdo_empty0 + 8u * uint32_t(bk.qs));     // ... this (Q, dO) pair
        if (qt == ntile - 1) { umma_commit(dkv_ready); ++kti; }
        if (kStream) umma_commit(dq_ready0 + 8u * uint32_t(g & 1));
        else if (j == nb - 1) umma_commit(dq_ready0);
        TRACEB(4, g);
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 12) {
    // ===================== math: thread = query row, the two warps of a lane quarter split the key columns ==========
    const int w = warp - 4, q = w & 3, half = w >> 2;
    const int r = q * 32 + lane;                           // row inside the query tile == TMEM lane
    const uint32_t t_lane = tmem_base + (uint32_t(q * 32) << 16);
    const float sl2 = 0.125f * 1.4426950408889634f;
    // per row: lse2 from the forward and D = sum_d dO O of the block's query tile; the NEXT block's are loaded while
    // this one is worked on
    float Ln = 0.f, Dn = 0.f;
    auto load_stats = [&](int g) {
      const Blk nx = block_of(g);
      const int qrow = nx.qt * BT + r;
      const bool ok = qrow < T;
      Ln = ok ? __ldg(lse2 + (int64_t(nx.item) * T + qrow)) : 0.f;
      Dn = ok ? __ldg(dsum + (int64_t(nx.item) * T + qrow)) : 0.f;
    };
    if (G > 0) load_stats(0);
    for (int blk = 0; blk < G; ++blk) {
      const Blk bk = block_of(blk);
      const int kt = bk.kt, qt = bk.qt;
      const float lse = Ln, Dq8 = Dn * 0.125f;
      if (blk + 1 < G) load_stats(blk + 1);
      {
        const int nk = ext(kt);
        {
          const uint32_t bph = uint32_t(blk & 1);
          const int qrow = qt * BT + r;
          const bool row_ok = qrow < T;
          const uint32_t ds_tile = sDS + uint32_t(blk & 1) * 2 * ATOM_BYTES;
          bool tiles_free = false;                         // waited for lazily: the first exponentials overlap the MMAs
          for (int hf = 0; hf < 2; ++hf) {                 // the block's two 64-key halves (TMEM double buffer)
            const int nkh = max(0, min(64, nk - 64 * hf));
            const int wcols = nkh / 2;                     // this warp's share of the half: 32, 8 (T = 197 tail) or 0
            const int cw = 64 * hf + half * wcols;         // first of this warp's columns
            mbar_wait(sdp_ready0 + 8u * hf, bph);
            if (w == 0 && lane == 0) TRACEB(hf == 0 ? 5 : 8, blk);
            tc_fence_after();
            // the block has no key or row past T (warp-uniform): no masking selects in the inner loop
            const bool full = __all_sync(0xffffffffu, row_ok) && kt * BT + 64 * hf + nkh <= T;
            // NN (32 or 8) key columns: scores and dP out of TMEM (the half is released at once), P and dS into the smem tiles
            auto chunk = [&](auto nn_tag, int c0, bool release) {
              constexpr int NN = decltype(nn_tag)::value;
              uint32_t sv[NN], dv[NN];
              if constexpr (NN == 32) {
                tmem_ld_32x32b_x32p(t_lane + COL_S + c0, sv);
                tmem_ld_32x32b_x32p(t_lane + COL_DP + c0, dv);
              } else {
                tmem_ld_32x32b_x8(t_lane + COL_S + c0, sv);
                tmem_ld_32x32b_x8(t_lane + COL_DP + c0, dv);
              }
              tmem_ld_wait();
              if (w == 0 && lane == 0) TRACEB(hf == 0 ? 12 : 13, blk);
              if (release) {                               // the warp's last values of this half are in registers:
                tc_fence_before();                         // the next block's half may be computed
                __syncwarp();
                if (lane == 0) mbar_arrive(sdp_free0 + 8u * hf);
              }
              uint32_t pk[NN / 2], dk[NN / 2];
#pragma unroll
              for (int e = 0; e < NN; e += 2) {
                float p0 = ex2_approx(fmaf(__uint_as_float(sv[e]), sl2, -lse));
                float p1 = ex2_approx(fmaf(__uint_as_float(sv[e + 1]), sl2, -lse));
                if (!full) {                               // rows / keys past T hold arbitrary bits
                  if (!(row_ok && kt * BT + c0 + e < T)) p0 = 0.f;
                  if (!(row_ok && kt * BT + c0 + e + 1 < T)) p1 = 0.f;
                }
                float d0 = p0 * fmaf(__uint_as_float(dv[e]), 0.125f, -Dq8);          // dS = P o (dP - D) / 8
                float d1 = p1 * fmaf(__uint_as_float(dv[e + 1]), 0.125f, -Dq8);
                if (!full) {
                  if (p0 == 0.f) d0 = 0.f;
                  if (p1 == 0.f) d1 = 0.f;
                }
                pk[e >> 1] = pack2<kDT>(p0, p1);
                dk[e >> 1] = pack2<kDT>(d0, d1);
              }
              if (!tiles_free) {
                if (w == 0 && lane == 0) TRACEB(6, blk);
                mbar_wait(p_free, bph ^ 1u);               // the previous block's dV MMAs have read the P tile
                mbar_wait(ds_free0 + 8u * uint32_t(blk & 1), (uint32_t(blk >> 1) & 1u) ^ 1u);   // dK / dQ of two blocks ago this dS tile
                tiles_free = true;
                if (w == 0 && lane == 0) TRACEB(7, blk);
              }
              if (w == 0 && lane == 0 && hf == 1) TRACEB(14, blk);
#pragma unroll
              for (int g = 0; g < NN / 8; ++g) {           // 8 key columns -> one 16-byte chunk of each tile
                const int c = c0 + g * 8;
                const uint32_t off = uint32_t(c >> 6) * ATOM_BYTES + uint32_t(r) * 128u + (uint32_t(((c & 63) >> 3) ^ (r & 7)) << 4);
                st_shared_v4(sP + off, pk[g * 4 + 0], pk[g * 4 + 1], pk[g * 4 + 2], pk[g * 4 + 3]);
                st_shared_v4(ds_tile + off, dk[g * 4 + 0], dk[g * 4 + 1], dk[g * 4 + 2], dk[g * 4 + 3]);
              }
            };
            if (wcols == 32) chunk(std::integral_constant<int, 32>{}, cw, true);
            else if (wcols > 0) {                          // 8, 16 or 24 columns (short sequences, the T = 197 tail)
              for (int c = 0; c < wcols; c += 8) chunk(std::integral_constant<int, 8>{}, cw + c, c + 8 >= wcols);
            } else {                                       // the half is empty
              __syncwarp();
              if (lane == 0) mbar_arrive(sdp_free0 + 8u * hf);
            }
          }
          if (w == 0 && lane == 0) TRACEB(15, blk);
          fence_proxy_async_smem();                        // generic-proxy tile writes -> the MMAs' async-proxy reads
          __syncwarp();
          if (lane == 0) mbar_arrive(pds_ready);
          if (w == 0 && lane == 0) TRACEB(9, blk);
        }
      }
    }
  } else if (warp >= 12) {
    // ===================== epilogue: dK / dV per key tile, dQ per item -> 16-bit rows of dqkv =====================
    const int q = warp & 3, r = q * 32 + lane;
    const uint32_t t_lane = tmem_base + (uint32_t(q * 32) << 16);
    const int64_t ld = 3 * int64_t(inner);
    auto store_row = [&](uint32_t col, uint16_t* dst) {    // 64 fp32 TMEM columns of this lane -> 64 16-bit values
      uint32_t v[64];
      tmem_ld_32x32b_x32p(t_lane + col, v);
      tmem_ld_32x32b_x32p(t_lane + col + 32, v + 32);
      tmem_ld_wait();
      if (dst != nullptr) {
        // 32-byte stores (STG.256): every lane writes its own row, so a warp-wide store touches 32 lines whatever its
        // width -- half as many requests as 16-byte ones in front of the math warps' tile stores in the same LSU
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t w[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) w[e] = pack2<kDT>(__uint_as_float(v[g * 16 + 2 * e]), __uint_as_float(v[g * 16 + 2 * e + 1]));
          asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + g * 16), "r"(w[0]), "r"(w[1]), "r"(w[2]),
                       "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
        }
      }
    };
    // dK / dV of a finished key tile -> 16-bit rows of dqkv
    auto drain_dkv = [&](int item, int kt, int kti) {
      const int b = item / heads, h = item - b * heads;
      uint16_t* rowbase = dqkv + int64_t(b) * T * ld + h * DH;
      const int key = kt * BT + r;
      mbar_wait(dkv_ready, uint32_t(kti & 1));
      tc_fence_after();
      store_row(COL_DK, key < T ? rowbase + int64_t(key) * ld + inner : nullptr);
      store_row(COL_DV, key < T ? rowbase + int64_t(key) * ld + 2 * inner : nullptr);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(dkv_free);
    };
    if constexpr (kStream) {
      // one dQ contribution per block: 64 fp32 columns of this lane's query row are ADDED into dq_acc [B T, heads 64]
      int kti = 0;
      for (int g = 0; g < G; ++g) {
        const Blk bk = block_of(g);
        const int b = bk.item / heads, h = bk.item - b * heads;
        const int qrow = bk.qt * BT + r;
        mbar_wait(dq_ready0 + 8u * uint32_t(g & 1), uint32_t(g >> 1) & 1u);
        tc_fence_after();
        uint32_t v[64];
        tmem_ld_32x32b_x32p(t_lane + COL_DQ + uint32_t(g & 1) * DH, v);
        tmem_ld_32x32b_x32p(t_lane + COL_DQ + uint32_t(g & 1) * DH + 32, v + 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(dq_free0 + 8u * uint32_t(g & 1));
        if (qrow < T) {
          float* dst = dq_acc + (int64_t(b) * T + qrow) * inner + h * DH;
#pragma unroll
          for (int c = 0; c < 64; c += 4)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + c), "f"(__uint_as_float(v[c])),
                         "f"(__uint_as_float(v[c + 1])), "f"(__uint_as_float(v[c + 2])), "f"(__uint_as_float(v[c + 3])) : "memory");
        }
        if (bk.qt == ntile - 1) { drain_dkv(bk.item, bk.kt, kti); ++kti; }
      }
    } else {
      int kti = 0;
      for (int it = 0; it < my_units; ++it) {
        const int item = int(blockIdx.x) + it * int(gridDim.x);
        const int b = item / heads, h = item - b * heads;
        uint16_t* rowbase = dqkv + int64_t(b) * T * ld + h * DH;
        for (int kt = 0; kt < ntile; ++kt, ++kti) drain_dkv(item, kt, kti);
        mbar_wait(dq_ready0, uint32_t(it & 1));
        tc_fence_after();
        for (int qt = 0; qt < ntile; ++qt) {
          const int qrow = qt * BT + r;
          store_row(COL_DQ + qt * DH, qrow < T ? rowbase + int64_t(qrow) * ld : nullptr);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(dq_free0);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

// D[item, t] = sum_d dO[b, t, h, d] O[b, t, h, d], item = b * heads + h: one warp per token row, eight lanes per head.
// The chunk loop has the same trip count on every lane (heads * 8 rounded up to the warp), so the full-mask shuffles
// always see all 32 lanes; lanes past the row's last chunk load nothing and store nothing.
template <int kDT>
__global__ void __launch_bounds__(256)
attn_bwd_rowdot_kernel(const uint16_t* __restrict__ d_out, const uint16_t* __restrict__ o_fwd, float* __restrict__ dsum,
                       int rows, int T, int heads) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = heads * DH;
  const int nchunk = heads * 8, nchunk_warp = (nchunk + 31) & ~31;
  for (int64_t row = int64_t(blockIdx.x) * 8 + warp; row < rows; row += int64_t(gridDim.x) * 8) {
    const int b = int(row / T), t = int(row - int64_t(b) * T);
    const uint4* dr = reinterpret_cast<const uint4*>(d_out + row * inner);
    const uint4* orow = reinterpret_cast<const uint4*>(o_fwd + row * inner);
    for (int c0 = 0; c0 < nchunk_warp; c0 += 32) {
      const int c = c0 + lane;                           // 16-byte chunk c = 8 values of head c / 8
      const bool active = c < nchunk;                    // uniform over each group of 8 lanes (nchunk % 8 == 0)
      float acc = 0.f;
      if (active) {
        const uint4 dv = __ldg(dr + c), ov = __ldg(orow + c);
        const uint32_t dd[4] = {dv.x, dv.y, dv.z, dv.w}, oo[4] = {ov.x, ov.y, ov.z, ov.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc = fmaf(to_f32<kDT>(uint16_t(dd[e] & 0xFFFFu)), to_f32<kDT>(uint16_t(oo[e] & 0xFFFFu)), acc);
          acc = fmaf(to_f32<kDT>(uint16_t(dd[e] >> 16)), to_f32<kDT>(uint16_t(oo[e] >> 16)), acc);
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if (active && (lane & 7) == 0) dsum[(int64_t(b) * heads + (c >> 3)) * T + t] = acc;
    }
  }
}

// fp32 dQ accumulator [rows, inner] -> the q third of dqkv (16 bits)
template <int kDT>
__global__ void __launch_bounds__(256)
dq_convert_kernel(const float* __restrict__ dq_acc, uint16_t* __restrict__ dqkv, int64_t rows, int inner) {
  const int per_row = inner >> 3;
  const int64_t total = rows * per_row;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = i / per_row;
    const int c = int(i - r * per_row) * 8;
    const float4 a = *reinterpret_cast<const float4*>(dq_acc + r * inner + c), b = *reinterpret_cast<const float4*>(dq_acc + r * inner + c + 4);
    uint4 o;
    o.x = pack2<kDT>(a.x, a.y); o.y = pack2<kDT>(a.z, a.w); o.z = pack2<kDT>(b.x, b.y); o.w = pack2<kDT>(b.z, b.w);
    *reinterpret_cast<uint4*>(dqkv + r * 3 * inner + c) = o;
  }
}

template <int kDT, bool kStream>
int launch_t(cudaStream_t st, const void* qkv, const void* d_out, void* dqkv, const float* lse2, const float* dsum,
             float* dq_acc, int batch, int T, int heads) {
  static PerDevice<bool> configured_on;
  if (bool& configured = configured_on.here(); !configured) {
    VB_CUDA(cudaFuncSetAttribute(attention_bwd_tc5_kernel<kDT, kStream>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL));
    configured = true;
  }
  const int inner = heads * DH;
  CUtensorMap tq, tdo;
  int rc;
  if ((rc = make_tmap_3d_16(&tq, qkv, batch, T, 3 * inner, 3 * inner, BT, kDT))) return rc;
  if ((rc = make_tmap_3d_16(&tdo, d_out, batch, T, inner, inner, BT, kDT))) return rc;
  const int items = batch * heads;
  const int64_t units = kStream ? int64_t(items) * ((T + BT - 1) / BT) : items;
  const int grid = int(units < sm_count() ? units : sm_count());
  VB_CUDA(launch_kernel(attention_bwd_tc5_kernel<kDT, kStream>, dim3(grid), dim3(NTHR), SMEM_TOTAL, st, 1, tq, tdo, lse2, dsum,
                        static_cast<uint16_t*>(dqkv), dq_acc, T, heads, items));
  VB_LAUNCH_CHECK("attention_bwd_tc5_kernel");
  return 0;
}

}  // namespace

#ifdef VITB200_TRACE
}  // namespace vb
extern "C" int vitb200_debug_attention_bwd_trace(long long* host, int n) {
  return cudaMemcpyFromSymbol(host, vb::g_trace_bwd, sizeof(long long) * (n < 16 * 64 ? n : 16 * 64)) == cudaSuccess ? 0 : -2;
}
namespace vb {
#endif

// fp32 dQ accumulator [rows, inner] -> the q third of dqkv (16-bit)
int launch_dq_convert(cudaStream_t st, const float* dq_acc, void* dqkv, int64_t rows, int inner, int dtype) {
  const unsigned cgrid = unsigned(std::min<int64_t>((rows * (inner / 8) + 255) / 256, int64_t(sm_count()) * 16));
  if (dtype == DT_F16) dq_convert_kernel<DT_F16><<<cgrid, 256, 0, st>>>(dq_acc, static_cast<uint16_t*>(dqkv), rows, inner);
  else if (dtype == DT_BF16) dq_convert_kernel<DT_BF16><<<cgrid, 256, 0, st>>>(dq_acc, static_cast<uint16_t*>(dqkv), rows, inner);
  else return fail(VITB200_ERR_INVALID, "attention_bwd: dtype must be bf16 or fp16");
  VB_LAUNCH_CHECK("dq_convert_kernel");
  return 0;
}

bool attention_bwd_tc5_supports(int T) { return T >= 1 && T <= ROWS_MAX; }

// D = rowsum(dO o O) per (image, head, token) into dsum [batch*heads, T]
int launch_attention_bwd_rowdot(cudaStream_t st, const void* d_out, const void* o_fwd, float* dsum, int batch, int T, int heads,
                                int dtype) {
  const int64_t rows = int64_t(batch) * T;
  const unsigned grid = unsigned(std::min<int64_t>((rows + 7) / 8, int64_t(sm_count()) * 16));
  if (dtype == DT_F16)
    attn_bwd_rowdot_kernel<DT_F16><<<grid, 256, 0, st>>>(static_cast<const uint16_t*>(d_out), static_cast<const uint16_t*>(o_fwd), dsum, int(rows), T, heads);
  else if (dtype == DT_BF16)
    attn_bwd_rowdot_kernel<DT_BF16><<<grid, 256, 0, st>>>(static_cast<const uint16_t*>(d_out), static_cast<const uint16_t*>(o_fwd), dsum, int(rows), T, heads);
  else return fail(VITB200_ERR_INVALID, "attention_bwd: dtype must be bf16 or fp16");
  VB_LAUNCH_CHECK("attn_bwd_rowdot_kernel");
  return 0;
}

int launch_attention_bwd_tc5(cudaStream_t st, const void* qkv, const void* d_out, void* dqkv, const float* lse2,
                             const float* dsum, int batch, int T, int heads, int dtype) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention_bwd: empty problem");
  if (!attention_bwd_tc5_supports(T)) return fail(VITB200_ERR_UNSUPPORTED, "attention_bwd_tc5: T > 208 needs the streamed form");
  if (lse2 == nullptr || dsum == nullptr) return fail(VITB200_ERR_INVALID, "attention_bwd_tc5: needs the forward's row log-sum-exp and D");
  if (dtype == DT_BF16) return launch_t<DT_BF16, false>(st, qkv, d_out, dqkv, lse2, dsum, nullptr, batch, T, heads);
  if (dtype == DT_F16) return launch_t<DT_F16, false>(st, qkv, d_out, dqkv, lse2, dsum, nullptr, batch, T, heads);
  return fail(VITB200_ERR_INVALID, "attention_bwd: dtype must be bf16 or fp16");
}

// any T: dK / dV from TMEM per (image, head, key tile), dQ summed into dq_acc (fp32 [batch * T, heads * 64], zeroed here)
// and converted into the q third of dqkv by a last pass
int launch_attention_bwd_tc5_stream(cudaStream_t st, const void* qkv, const void* d_out, void* dqkv, const float* lse2,
                                    const float* dsum, float* dq_acc, int batch, int T, int heads, int dtype) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention_bwd: empty problem");
  if (lse2 == nullptr || dsum == nullptr || dq_acc == nullptr)
    return fail(VITB200_ERR_INVALID, "attention_bwd_tc5: the streamed form needs lse2, D and the fp32 dQ buffer");
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(VITB200_ERR_INVALID, "attention_bwd: dtype must be bf16 or fp16");
  const int64_t rows = int64_t(batch) * T;
  const int inner = heads * DH;
  VB_CUDA(cudaMemsetAsync(dq_acc, 0, size_t(rows) * inner * sizeof(float), st));
  int rc = dtype == DT_BF16 ? launch_t<DT_BF16, true>(st, qkv, d_out, dqkv, lse2, dsum, dq_acc, batch, T, heads)
                            : launch_t<DT_F16, true>(st, qkv, d_out, dqkv, lse2, dsum, dq_acc, batch, T, heads);
  if (rc) return rc;
  return launch_dq_convert(st, dq_acc, dqkv, rows, inner, dtype);
}

}  // namespace vb
