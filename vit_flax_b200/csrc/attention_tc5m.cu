// attention_tc5m.cu -- K4 for long sequences (T > 208: ViT-H/14 T = 257, 512-px ViT-L/16 T = 1025):
// the tcgen05 / TMEM attention of attention_tc5.cu with the keys streamed in blocks of KP and an
// online softmax.
//
//   out = softmax(Q K^T * 64^-0.5) V   per (image, head)                        vit.py:69-79
//
// One work item = (image, head, 128-query tile); it walks the nkb = ceil(T / KP) key blocks.
// Same 16-warp layout as the one-block kernel: TMA producer, one MMA issuer per TMEM slot (warps
// 1 and 3), two softmax groups (thread = query row = TMEM lane), four epilogue warps.  A softmax
// group owns one item at a time and TMEM slot `grp`:
//   slot s:  S_j (fp32, KP columns) then P_j (16-bit pairs, KP/2 columns)   at column s*KP
//            O   (fp32, 64 columns), the item's accumulator                 at column 2*KP + s*64
// Per key block j:  S_j = Q K_j^T  ->  block max, running max m, rescale factor a = 2^((m_old -
// m_new) * scale*log2e)  ->  if any row of the warp moved its max: O *= a through
// tcgen05.ld / tcgen05.st (after PV_{j-1} has completed)  ->  P_j = 2^(S_j*scale*log2e - m_new*...)
// over S_j, running sum l = l*a + sum(P_j)  ->  O += P_j V_j (accumulate).  After the last block the
// epilogue warps pull O into registers, scale by 1/l and TMA-store the tile (rows >= T clipped).
// Keys >= T arrive as zero-filled K rows (score 0): they are masked to -inf in the last block.
// K_j / V_j stream through a 3-deep ring per item (they are L2-resident: 2*T*128 B per
// (image, head), re-read by its ceil(T/128) q tiles); Q has one stage per slot.
#include <cstdlib>

#include "common.h"
#include "ptx.cuh"

namespace vb {

namespace {

constexpr int DH = 64;
constexpr int QT = 128;                 // queries per work item (UMMA M)
constexpr int NT = 512;                 // 4 service warps, 2 x 4 softmax, 4 epilogue
constexpr int Q_BYTES = QT * 128;
constexpr int O_BYTES = QT * 128;
constexpr int KS = 3;                   // K / V ring depth (key blocks in flight)

template <int KP>
struct SmemM {
  static constexpr int KV_BYTES = KP * 128;
  static constexpr int OFF_Q = 0;                             // 2 stages (one per slot)
  static constexpr int OFF_K = OFF_Q + 2 * Q_BYTES;
  static constexpr int OFF_V = OFF_K + KS * KV_BYTES;
  static constexpr int OFF_O = OFF_V + KS * KV_BYTES;         // 2 staging buffers
  static constexpr int OFF_BAR = OFF_O + 2 * O_BYTES;         // 32 mbarrier slots
  static constexpr int OFF_INV = OFF_BAR + 256;               // float [4][128]
  static constexpr int TOTAL = OFF_INV + 4 * 128 * 4 + 1024 /*align slack*/;
  static_assert(KV_BYTES % 1024 == 0, "K/V stage must keep 1024-byte alignment");
  static_assert(TOTAL <= 232448, "shared memory budget");
  static_assert(2 * KP + 2 * DH <= 512, "TMEM budget: two score slots + two accumulators");
};

// NN (32 or 16) score columns in registers -> p = exp2(s*sl2 + mneg), fp32 partial sums, 16-bit pairs
template <int kDT, int NN, bool kMask>
__device__ __forceinline__ void exp_chunk(uint32_t* r, uint32_t* pp, int c0, int nvalid,
                                          unsigned long long sl2x2, unsigned long long mnegx2,
                                          unsigned long long& la, unsigned long long& lb) {
  if constexpr (kMask) {
#pragma unroll
    for (int j = 0; j < NN; ++j)
      if (c0 + j >= nvalid) r[j] = __float_as_uint(-INFINITY);
  }
#pragma unroll
  for (int j = 0; j < NN / 2; ++j) {
    float a0, a1;
    unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])), sl2x2, mnegx2), a0, a1);
    const float p0 = ex2_approx(a0), p1 = ex2_approx(a1);
    if (j & 1) lb = add_f32x2(lb, pack_f32x2(p0, p1));
    else la = add_f32x2(la, pack_f32x2(p0, p1));
    pp[j] = pack2<kDT>(p0, p1);
  }
}

// Wait for turn `turn` on the hand-off barrier: phases complete in turn order, one per turn, when
// the 4 warps of the acting group arrive.  A parity wait tells "phase turn-1 done" from "not done"
// only if phase turn-2 (this group's previous turn) is known to be complete: every arrive is
// therefore followed by a group barrier (pass_turn), so that no warp tests for the partner's turn
// while its own group's phase is still open.
__device__ __forceinline__ void wait_turn(uint32_t bar, uint32_t turn) {
  mbar_wait(bar, (turn & 1u) ^ 1u);
}
__device__ __forceinline__ void pass_turn(uint32_t bar, int grp, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
  named_bar_sync(2 + grp, 128);
}

template <int kDT, int KP>
__global__ void __launch_bounds__(NT, 1)
attention_tc5m_kernel(const __grid_constant__ CUtensorMap tmQ,    // qkv [B,T,3I], box 128 rows
                      const __grid_constant__ CUtensorMap tmKV,   // qkv [B,T,3I], box KP rows
                      const __grid_constant__ CUtensorMap tmO,    // out [B,T,I],  box 128 rows
                      int T, int heads, int nqt, int nkb, int items, int turns, float* __restrict__ lse_out) {
  using L = SmemM<KP>;
  constexpr uint32_t O_COL = 2 * KP;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQ = base + L::OFF_Q, sK = base + L::OFF_K, sV = base + L::OFF_V, sO = base + L::OFF_O;
  const uint32_t bars = base + L::OFF_BAR;
  auto q_full = [&](int s) { return bars + 8u * (0 + s); };    // [2]
  auto q_empty = [&](int s) { return bars + 8u * (2 + s); };   // [2]
  auto k_full = [&](int s) { return bars + 8u * (4 + s); };    // [KS]
  auto k_empty = [&](int s) { return bars + 8u * (7 + s); };
  auto v_full = [&](int s) { return bars + 8u * (10 + s); };
  auto v_empty = [&](int s) { return bars + 8u * (13 + s); };
  auto s_ready = [&](int s) { return bars + 8u * (16 + s); };  // [2 slots]
  auto p_ready = [&](int s) { return bars + 8u * (18 + s); };
  auto pv_done = [&](int s) { return bars + 8u * (20 + s); };
  auto o_ready = [&](int s) { return bars + 8u * (22 + s); };
  auto o_free = [&](int s) { return bars + 8u * (24 + s); };
  const uint32_t xu_done = bars + 8u * 26;                     // exponential phases take turns
  const uint32_t tmem_slot = bars + 8u * 27;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + L::OFF_BAR + 8 * 27);
  float* inv_sh = reinterpret_cast<float*>(gbase + L::OFF_INV);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = heads * DH;
  const int64_t first = int64_t(blockIdx.x) * items / gridDim.x;
  const int64_t last = int64_t(blockIdx.x + 1) * items / gridDim.x;
  const int n = int(last - first);
  // K/V ring entries are numbered in the order the two issuers consume them: the blocks of items
  // 2p and 2p+1 (one per slot) interleave, an unpaired last item runs alone.
  auto ring_seq = [&](int i, int j) {
    const bool paired = (i | 1) < n;
    return (i >> 1) * 2 * nkb + (paired ? 2 * j + (i & 1) : j);
  };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmQ);
    prefetch_tmap(&tmKV);
    prefetch_tmap(&tmO);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(q_full(s), 1);
      mbar_init(q_empty(s), 1);
      mbar_init(s_ready(s), 1);
      mbar_init(p_ready(s), 4);
      mbar_init(pv_done(s), 1);
      mbar_init(o_ready(s), 1);
      mbar_init(o_free(s), 4);
    }
    for (int s = 0; s < KS; ++s) {
      mbar_init(k_full(s), 1);
      mbar_init(k_empty(s), 1);
      mbar_init(v_full(s), 1);
      mbar_init(v_empty(s), 1);
    }
    mbar_init(xu_done, 4);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<1>(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_launch_dependents();
  pdl_wait();                // the to_qkv GEMM has completed

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      for (int i0 = 0; i0 < n; i0 += 2) {
        const int ni = (i0 + 1 < n) ? 2 : 1;             // items of this pair
        int bb[2], hh[2];
        for (int d = 0; d < ni; ++d) {
          const int i = i0 + d;
          const int64_t item = first + i;
          const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
          bb[d] = bh / heads;
          hh[d] = bh - bb[d] * heads;
          mbar_wait(q_empty(d), ((i >> 1) & 1) ^ 1u);
          mbar_arrive_expect_tx(q_full(d), Q_BYTES);
          tma_load_3d(sQ + d * Q_BYTES, &tmQ, q_full(d), hh[d] * DH, qt * QT, bb[d]);
        }
        for (int j = 0; j < nkb; ++j) {
          for (int d = 0; d < ni; ++d) {
            const int e = ring_seq(i0 + d, j), es = e % KS;
            const uint32_t eph = (e / KS) & 1;
            mbar_wait(k_empty(es), eph ^ 1u);
            mbar_arrive_expect_tx(k_full(es), L::KV_BYTES);
            tma_load_3d(sK + es * L::KV_BYTES, &tmKV, k_full(es), inner + hh[d] * DH, j * KP, bb[d]);
            mbar_wait(v_empty(es), eph ^ 1u);
            mbar_arrive_expect_tx(v_full(es), L::KV_BYTES);
            tma_load_3d(sV + es * L::KV_BYTES, &tmKV, v_full(es), 2 * inner + hh[d] * DH, j * KP, bb[d]);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 3) {
    // ===================== MMA issuers: warp 1 drives slot 0, warp 3 slot 1 =====================
    if (elect_one()) {
      constexpr int fmt = kDT == DT_F16 ? 0 : 1;
      constexpr uint32_t idesc_s = umma_idesc_16(QT, KP, fmt, 0);   // B = K, K-major
      constexpr uint32_t idesc_o = umma_idesc_16(QT, DH, fmt, 1);   // B = V, MN-major
      const int s = warp == 1 ? 0 : 1;
      const uint32_t d_s = tmem_base + s * KP, d_o = tmem_base + O_COL + s * DH;
      for (int i = s; i < n; i += 2) {
        const uint32_t iph = (i >> 1) & 1;
        mbar_wait(q_full(s), iph);
        for (int j = 0; j < nkb; ++j) {
          const int e = ring_seq(i, j), es = e % KS;
          const uint32_t eph = (e / KS) & 1;
          const uint32_t uph = uint32_t((i >> 1) * nkb + j) & 1u;   // block count on this slot
          // S_j = Q K_j^T (the slot's previous P was consumed by this thread's previous PV)
          mbar_wait(k_full(es), eph);
          tc_fence_after();
          const uint32_t q0 = sQ + s * Q_BYTES, k0 = sK + es * L::KV_BYTES;
#pragma unroll
          for (int k = 0; k < DH / 16; ++k)
            umma_bf16_ss<1>(d_s, umma_desc_k_sw128(q0 + k * 32), umma_desc_k_sw128(k0 + k * 32), idesc_s,
                            k != 0 ? 1u : 0u);
          umma_commit(k_empty(es));
          if (j == nkb - 1) umma_commit(q_empty(s));
          umma_commit(s_ready(s));
          // O (+)= P_j V_j
          mbar_wait(p_ready(s), uph);
          mbar_wait(v_full(es), eph);
          if (j == 0) mbar_wait(o_free(s), iph ^ 1u);     // the previous item's O has been read out
          tc_fence_after();
          const uint32_t v0 = sV + es * L::KV_BYTES;
#pragma unroll
          for (int kk = 0; kk < KP / 16; ++kk)
            umma_bf16_ts(d_o, d_s + kk * 8, umma_desc_mn_sw128(v0 + kk * 2048), idesc_o,
                         (j | kk) != 0 ? 1u : 0u);
          umma_commit(v_empty(es));
          umma_commit(pv_done(s));
          if (j == nkb - 1) umma_commit(o_ready(s));
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 12) {
    // ===================== softmax (two independent groups) =====================
    const int w = warp - 4;
    const int q = w & 3;                  // TMEM lane quarter (== warp % 4)
    const int grp = w >> 2;               // group == TMEM slot
    const int row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + (uint32_t(q * 32) << 16);
    const uint32_t t_slot = t_lane + uint32_t(grp * KP);
    const uint32_t t_o = t_lane + O_COL + uint32_t(grp * DH);
    const float sl2 = 0.125f * 1.4426950408889634f;   // dim_head^-0.5 * log2(e)   (vit.py:66)
    constexpr int NFULL = KP / 32, TAIL = KP % 32;
    static_assert(TAIL == 0 || TAIL == 16, "key block = n*32 (+16)");

    for (int i = grp; i < n; i += 2) {
      const int64_t item = first + i;
      const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
      const bool active = qt * QT + q * 32 < T;          // warp-uniform: any valid query row here?
      float m = -INFINITY, l = 0.f;
      for (int j = 0; j < nkb; ++j) {
        const uint32_t u = uint32_t((i >> 1) * nkb + j);
        const uint32_t turn = 2u * u + uint32_t(grp);      // position in the alternating order
        const int nvalid = T - j * KP;                    // valid keys of this block (>= KP: all)
        mbar_wait(s_ready(grp), u & 1u);
        tc_fence_after();
        if (active) {
          uint32_t r[2][32];
          // ---- pass 1: block max ----
          float bm = -INFINITY;
          tmem_ld_32x32b_x32p(t_slot, r[0]);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < NFULL; ++c) {
            if (c + 1 < NFULL) tmem_ld_32x32b_x32p(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
            else if (TAIL) tmem_ld_32x32b_x16(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
            uint32_t* rc = r[c & 1];
            if (c * 32 + 32 > nvalid) {                   // warp-uniform: only chunks past T pay
#pragma unroll
              for (int k = 0; k < 32; ++k)
                if (c * 32 + k >= nvalid) rc[k] = __float_as_uint(-INFINITY);
            }
#pragma unroll
            for (int k = 0; k < 32; k += 2)
              bm = fmaxf(bm, fmaxf(__uint_as_float(rc[k]), __uint_as_float(rc[k + 1])));
            if (c + 1 < NFULL || TAIL) tmem_ld_wait();
          }
          if constexpr (TAIL != 0) {
            uint32_t* rc = r[NFULL & 1];
#pragma unroll
            for (int k = 0; k < 16; ++k)
              if (NFULL * 32 + k >= nvalid) rc[k] = __float_as_uint(-INFINITY);
#pragma unroll
            for (int k = 0; k < 16; k += 2)
              bm = fmaxf(bm, fmaxf(__uint_as_float(rc[k]), __uint_as_float(rc[k + 1])));
          }
          // ---- running max; rescale the accumulator and the running sum when a row's max moved ----
          const float m_new = fmaxf(m, bm);
          if (j > 0) {
            const float alpha = ex2_approx((m - m_new) * sl2);      // 1 when the max did not move
            l *= alpha;
            mbar_wait(pv_done(grp), (u - 1u) & 1u);                 // PV_{j-1} complete: O is stable
            tc_fence_after();
            if (__any_sync(0xffffffffu, m_new > m)) {
              uint32_t o[64];
              tmem_ld_32x32b_x32p(t_o, o);
              tmem_ld_32x32b_x32p(t_o + 32, o + 32);
              tmem_ld_wait();
#pragma unroll
              for (int k = 0; k < 64; ++k) o[k] = __float_as_uint(__uint_as_float(o[k]) * alpha);
              tmem_st_32x32b_x16(t_o, o);
              tmem_st_32x32b_x16(t_o + 16, o + 16);
              tmem_st_32x32b_x16(t_o + 32, o + 32);
              tmem_st_32x32b_x16(t_o + 48, o + 48);
            }
          }
          m = m_new;
          // The exponential phases of the two groups take turns, block by block (see attention_tc5.cu:
          // free-running groups fall into step and idle the XU pipe while both wait for their MMAs).
          if (turns) wait_turn(xu_done, turn);
          // ---- pass 2: p = exp2((s - m) * scale * log2e); l += sum(p); P -> TMEM over S ----
          const float mneg = -m * sl2;
          const unsigned long long sl2x2 = pack_f32x2(sl2, sl2), mnegx2 = pack_f32x2(mneg, mneg);
          unsigned long long la = pack_f32x2(0.f, 0.f), lb = la;
          tmem_ld_32x32b_x32p(t_slot, r[0]);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < NFULL; ++c) {
            if (c + 1 < NFULL) tmem_ld_32x32b_x32p(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
            else if (TAIL) tmem_ld_32x32b_x16(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
            uint32_t pp[16];
            if (c * 32 + 32 > nvalid) exp_chunk<kDT, 32, true>(r[c & 1], pp, c * 32, nvalid, sl2x2, mnegx2, la, lb);
            else exp_chunk<kDT, 32, false>(r[c & 1], pp, c * 32, nvalid, sl2x2, mnegx2, la, lb);
            if (c + 1 < NFULL || TAIL) tmem_ld_wait();
            tmem_st_32x32b_x16(t_slot + c * 16, pp);
          }
          if constexpr (TAIL != 0) {
            uint32_t pp[8];
            exp_chunk<kDT, 16, true>(r[NFULL & 1], pp, NFULL * 32, nvalid, sl2x2, mnegx2, la, lb);
            tmem_st_32x32b_x8(t_slot + NFULL * 16, pp);
          }
          float l0, l1;
          unpack_f32x2(add_f32x2(la, lb), l0, l1);
          l += l0 + l1;
          if (j == nkb - 1) {
            inv_sh[(i & 3) * 128 + row] = 1.0f / l;   // for the epilogue warps
            // training: the row's log-sum-exp in the log2 domain (m is the running max of the raw scores), for the adjoint
            if (lse_out != nullptr && qt * QT + row < T) lse_out[int64_t(bh) * T + qt * QT + row] = m * sl2 + __log2f(l);
          }
          tmem_st_wait();
        } else if (turns) {
          wait_turn(xu_done, turn);
        }
        if (turns) pass_turn(xu_done, grp, lane);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_ready(grp));
      }
    }
    if (turns && grp == 1 && (n & 1)) {
      // the last item has no partner: group 1 passes its turns on so group 0 is never left waiting
      for (int j = 0; j < nkb; ++j) {
        const uint32_t turn = 2u * uint32_t((n >> 1) * nkb + j) + 1u;
        wait_turn(xu_done, turn);
        pass_turn(xu_done, grp, lane);
      }
    }
  } else if (warp >= 12) {
    // ===================== epilogue: O / rowsum -> 16-bit -> swizzled smem -> TMA store ==========
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool leader = (q == 0 && lane == 0);
    const uint32_t t_lane = tmem_base + (uint32_t(q * 32) << 16);
    for (int i = 0; i < n; ++i) {
      const int s = i & 1;
      const uint32_t ph = (i >> 1) & 1;
      const int64_t item = first + i;
      const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
      const int b = bh / heads, h = bh - b * heads;
      const bool active = qt * QT + q * 32 < T;
      const uint32_t sOi = sO + uint32_t(i & 1) * O_BYTES;
      mbar_wait(o_ready(s), ph);                         // last PV of item i done (issued after the
      tc_fence_after();                                  // group's final p_ready: 1/l is visible)
      uint32_t o[64];
      float inv = 0.f;
      if (active) {
        tmem_ld_32x32b_x32p(t_lane + O_COL + s * DH, o);
        tmem_ld_32x32b_x32p(t_lane + O_COL + s * DH + 32, o + 32);
        inv = inv_sh[(i & 3) * 128 + row];
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free(s));             // O is in registers: the slot's next item may start
      if (active) {
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          st_shared_v4(sOi + uint32_t(row) * 128u + (uint32_t(g ^ (row & 7)) << 4),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 0]) * inv, __uint_as_float(o[g * 8 + 1]) * inv),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 2]) * inv, __uint_as_float(o[g * 8 + 3]) * inv),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 4]) * inv, __uint_as_float(o[g * 8 + 5]) * inv),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 6]) * inv, __uint_as_float(o[g * 8 + 7]) * inv));
        }
      }
      fence_proxy_async_smem();
      if (leader) tma_store_wait_read<0>();              // store of item i-1 (other buffer) has been read out
      named_bar_sync(1, 128);
      if (leader) {
        tma_store_3d(&tmO, sOi, h * DH, qt * QT, b);     // rows >= T are clipped by the tensor map
        tma_store_commit();
      }
    }
    if (leader) tma_store_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

int attn_m_turns() {   // VITB200_ATTN_TURNS=0: free-running groups (A/B tests)
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VITB200_ATTN_TURNS");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v;
}

template <int kDT, int KP>
int launch_m(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads, float* lse, int q_tiles) {
  using L = SmemM<KP>;
  static PerDevice<bool> configured_on;   // the smem opt-in is per (function, device)
  if (bool& configured = configured_on.here(); !configured) {
    VB_CUDA(cudaFuncSetAttribute(attention_tc5m_kernel<kDT, KP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 L::TOTAL));
    configured = true;
  }
  const int inner = heads * DH;
  CUtensorMap tq, tkv, to;
  int rc;
  if ((rc = make_tmap_3d_16(&tq, qkv, batch, T, 3 * inner, 3 * inner, QT, kDT))) return rc;
  if ((rc = make_tmap_3d_16(&tkv, qkv, batch, T, 3 * inner, 3 * inner, KP, kDT))) return rc;
  if ((rc = make_tmap_3d_16(&to, out, batch, T, inner, inner, QT, kDT))) return rc;
  // nqt q tiles per (image, head): fewer than ceil(T / QT) computes only the first query rows of every image
  const int nqt = q_tiles > 0 && q_tiles < ceil_div(T, QT) ? q_tiles : ceil_div(T, QT), nkb = ceil_div(T, KP);
  const int64_t items64 = int64_t(batch) * heads * nqt;
  if (items64 > 0x7fffffff / nkb) return fail(VITB200_ERR_INVALID, "attention: too many work items");
  const int items = int(items64);
  const int grid = items < sm_count() ? items : sm_count();
  VB_CUDA(launch_kernel(attention_tc5m_kernel<kDT, KP>, dim3(grid), dim3(NT), L::TOTAL, stream, 1,
                        tq, tkv, to, T, heads, nqt, nkb, items, attn_m_turns(), lse));
  VB_LAUNCH_CHECK("attention_tc5m_kernel");
  return 0;
}

template <int kDT>
int launch_m_dt(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads, float* lse, int q_tiles) {
  // two blocks of 144 cover T <= 288 (ViT-H/14: 257) with less padding than two of 192
  if (T <= 288) return launch_m<kDT, 144>(stream, qkv, out, batch, T, heads, lse, q_tiles);
  return launch_m<kDT, 192>(stream, qkv, out, batch, T, heads, lse, q_tiles);
}

}  // namespace

int launch_attention_tc5m(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads,
                          int dtype, float* lse, int q_tiles) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention: empty problem");
  if (dtype == DT_BF16) return launch_m_dt<DT_BF16>(stream, qkv, out, batch, T, heads, lse, q_tiles);
  if (dtype == DT_F16) return launch_m_dt<DT_F16>(stream, qkv, out, batch, T, heads, lse, q_tiles);
  return fail(VITB200_ERR_INVALID, "attention: dtype must be bf16 or fp16");
}

}  // namespace vb
