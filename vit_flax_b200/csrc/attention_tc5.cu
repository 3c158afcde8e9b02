// attention_tc5.cu -- K4: fused attention on tcgen05 / TMEM for sequences that fit one key block
// (T <= 208 tokens: every 224-px /16 config, i.e. ViT-B/16 and ViT-L/16).
//
//   out = softmax(Q K^T * 64^-0.5) V   per (image, head)                        vit.py:69-79
//
// One work item = (image, head, 128-query tile).  Persistent CTAs, 16 warps:
//   warp 0  lane 0 : TMA producer.  Q tile, K, V boxes are cut straight out of the to_qkv output
//                    viewed as [B, T, 3I] (the split / head rearranges of vit.py:69-71 are
//                    coordinates); rows >= T are out of bounds of the image and arrive as zeros.
//                    K and V of an (image, head) are loaded once and shared by its q tiles (2-deep
//                    ring); Q has a 4-deep ring, so loads run one to two items ahead of the MMAs.
//   warps 1, 3     : tcgen05.mma issuers, one per TMEM slot (lane 0 each, blocking mbarrier waits):
//                      S = Q K^T  (M=128, N=KP, K=64; SS operands)
//                      O = P V    (M=128, N=64,  K=KP; P from TMEM, V MN-major), issued in PARTS of 64 keys
//                      as the softmax group publishes them (p_part barriers): the product runs UNDER the
//                      exponentials instead of behind them, so a slot is busy from S(i) to the end of pass 2
//                      plus one short tail, and S(i+2) -- queued right behind the last part, MMAs of one
//                      thread execute in order -- is ready long before the group's next turn.
//   warp 2         : TMEM allocator: two slots of KP columns (S fp32, then P as 16-bit pairs over
//                    the first KP/2 columns) + one 64-column O accumulator shared by both slots.
//   warps 4..7     : softmax group 0 -- items 0, 2, 4, ... of this CTA (slot 0)
//   warps 8..11    : softmax group 1 -- items 1, 3, 5, ... of this CTA (slot 1)
//   warps 12..15   : epilogue: O -> registers (frees the accumulator for the next PV), x 1/rowsum,
//                    16-bit, swizzled smem staging (2 buffers) -> TMA store, rows >= T clipped.
// A softmax thread owns one query row (= one TMEM lane): row max and row sum need no exchange.
// Pass 1 streams the score row out of TMEM for the max, pass 2 streams it again (TMEM reads are
// cheap), exponentiates, sums in fp32 and writes P back over S with tcgen05.st; 1/rowsum goes to
// the epilogue warps through shared memory.
// What bounds it (measured; profiles/r01_attention.md, profiles/r02_attention.md).  XU work -- ex2 at 8 cycles per
// warp instruction and SMSP plus the fp32 -> 16-bit pack F2FP at 4: 20 cycles per pair of scores -- is 2.08 k cycles
// per item; the tensor side is 0.64 k (S: four dependent UTCHMMA of N = 208) + 0.73 k (P V: thirteen of N = 64, paced by
// the ~50-cycle issue cost of one tcgen05.mma, not by the pipe: profiles/microbench/mma_chain.cu); the kernel runs at
// ~3.0 k cycles per item (79 us per launch at ViT-B/16 batch 256) because a TMEM slot goes round a LATENCY loop -- S 0.6-1.1 k, pass 1 0.7 k, pass 2 2.6 k (a
// single warp issues in order and ptxas batches a chunk's MUFUs apart from its FFMA2 / FADD2 / F2FP work), store drain
// 0.4 k, last P V part + next S issue 0.5-1.0 k -- and 512 TMEM columns hold two slots, no more.  The exponential phases
// of the two groups are offset per SMSP (xu_done[q]: warp q hands over to warp q of the other group one chunk before
// it finishes; free-running or earlier hand-offs measure the same within 2 %, strict alternation is 12 % slower).
// Round-2 experiments that did NOT pay and were removed: all eight softmax warps on every item with the key columns
// split between the two warps of a lane quarter (no phase overlap between items: 118 us against 84 at the time); the bf16 pack on
// the integer pipe (add 0x8000 + PRMT: 97 against 88 us -- the softmax warps are short of issue slots, not of XU
// cycles); hand-ordered volatile-asm interleaving of MUFU and FMA work (ptxas reschedules it to the same SASS); round
// 1's polynomial ex2 on the FMA pipe.
// Warps whose 32 query rows are all >= T (the last quarter of the 69-row tail tile at T = 197)
// skip their softmax: rows of an MMA are independent and those rows are never stored.
// The [B,h,T,T] score tensor of vit.py:73-75 never reaches HBM.
#include <cstdlib>

#include "common.h"
#include "ptx.cuh"

namespace vb {

#ifdef VITB200_TRACE
// debug timeline of CTA 0: g_trace[event][item] = clock64 at the event (profiles/trace_attention.py)
__device__ long long g_trace[12][64];
#define TRACE(ev, i) do { if (blockIdx.x == 0 && (i) < 64) g_trace[ev][i] = clock64(); } while (0)
#else
#define TRACE(ev, i) do { } while (0)
#endif

namespace {

constexpr int DH = 64;
constexpr int QT = 128;                 // queries per work item (UMMA M)
constexpr int NT = 512;                 // threads per CTA: 4 service warps, 2 x 4 softmax, 4 epilogue
constexpr int Q_BYTES = QT * 128;       // 16 KB
constexpr int O_BYTES = QT * 128;       // 16 KB staging for the TMA store (one per softmax group)

constexpr int QS = 4;                   // Q ring depth (one tile per item)
constexpr int KS = 2;                   // K/V ring depth (one entry per (image, head), shared by its q tiles)

template <int KP>
struct Smem {
  static constexpr int KV_BYTES = KP * 128;
  static constexpr int OFF_Q = 0;
  static constexpr int OFF_K = OFF_Q + QS * Q_BYTES;
  static constexpr int OFF_V = OFF_K + KS * KV_BYTES;
  static constexpr int OFF_O = OFF_V + KS * KV_BYTES;
  static constexpr int OFF_BAR = OFF_O + 2 * O_BYTES;        // 2 staging buffers; then 64 mbarrier slots
  static constexpr int OFF_INV = OFF_BAR + 512;              // float [4][128]: 1/rowsum, by item parity mod 4
  static constexpr int TOTAL = OFF_INV + 4 * 128 * 4 + 1024 /*align slack*/;
  static_assert(KV_BYTES % 1024 == 0, "K/V stage must keep 1024-byte alignment");
  static_assert(TOTAL <= 232448, "shared memory budget");
};

// NN (32 or 16) score columns of this thread's row, already in registers:
// p = exp2(s*sl2 + mneg) -> fp32 partial sums (la/lb) -> 16-bit P pairs.  kMask: the chunk may reach
// past T (keys >= T are zero-filled K rows: score 0, not -inf, so they are forced to -inf here).
template <int kDT, int NN, bool kMask>
__device__ __forceinline__ void softmax_chunk(uint32_t* r, uint32_t* pp, int c0, int T,
                                              unsigned long long sl2x2, unsigned long long mnegx2,
                                              unsigned long long& la, unsigned long long& lb) {
  if constexpr (kMask) {
#pragma unroll
    for (int j = 0; j < NN; ++j)
      if (c0 + j >= T) r[j] = __float_as_uint(-INFINITY);
  }
#pragma unroll
  for (int j = 0; j < NN / 2; ++j) {
    const unsigned long long a2 =
        fma_f32x2(pack_f32x2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])), sl2x2, mnegx2);
    float a0, a1;
    unpack_f32x2(a2, a0, a1);
    const float p0 = ex2_approx(a0), p1 = ex2_approx(a1);
    if (j & 1) lb = add_f32x2(lb, pack_f32x2(p0, p1));
    else la = add_f32x2(la, pack_f32x2(p0, p1));
    pp[j] = pack2<kDT>(p0, p1);
  }
}

template <int kDT, int KP>
__global__ void __launch_bounds__(NT, 1)
attention_tc5_kernel(const __grid_constant__ CUtensorMap tmQ,    // qkv [B,T,3I], box 128 rows
                     const __grid_constant__ CUtensorMap tmKV,   // qkv [B,T,3I], box KP rows
                     const __grid_constant__ CUtensorMap tmO,    // out [B,T,I],  box 128 rows
                     int T, int heads, int nqt, int items, int turns, float* __restrict__ lse_out) {
  using L = Smem<KP>;
  // TMEM columns: slot s holds S (fp32, KP columns) then P (16-bit pairs, KP/2 columns) of the
  // item in flight on it; one O accumulator (64 columns) is shared by both slots.
  constexpr uint32_t SLOT_COLS = KP <= 128 ? 128 : 208;
  constexpr uint32_t O_COL = 2 * SLOT_COLS;
  static_assert(O_COL + DH <= 512, "TMEM budget");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQ = base + L::OFF_Q, sK = base + L::OFF_K, sV = base + L::OFF_V, sO = base + L::OFF_O;
  const uint32_t bars = base + L::OFF_BAR;
  auto q_full = [&](int s) { return bars + 8u * (0 + s); };    // [QS]
  auto q_empty = [&](int s) { return bars + 8u * (4 + s); };   // [QS]
  auto k_full = [&](int s) { return bars + 8u * (8 + s); };    // [KS]
  auto v_full = [&](int s) { return bars + 8u * (10 + s); };
  auto k_empty = [&](int s) { return bars + 8u * (12 + s); };
  auto v_empty = [&](int s) { return bars + 8u * (14 + s); };
  auto s_ready = [&](int s) { return bars + 8u * (16 + s); };  // [2 TMEM slots]
  auto o_ready = [&](int s) { return bars + 8u * (20 + s); };
  const uint32_t o_free = bars + 8u * 22;
  auto p_part = [&](int s, int g) { return bars + 8u * (32 + 4 * s + g); };   // [2 slots][<= 4 parts of 64 keys]
  auto xu_done = [&](int q) { return bars + 8u * (40 + q); };  // [4 SMSPs]: exponential phases take turns (see below)
  const uint32_t tmem_slot = bars + 8u * 24;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + L::OFF_BAR + 8 * 24);
  float* inv_sh = reinterpret_cast<float*>(gbase + L::OFF_INV);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = heads * DH;
  if (turns < 0) turns = KP / 32 - 1 > 0 ? KP / 32 - 1 : 1;
  const int64_t first = int64_t(blockIdx.x) * items / gridDim.x;
  const int64_t last = int64_t(blockIdx.x + 1) * items / gridDim.x;
  const int n = int(last - first);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmQ);
    prefetch_tmap(&tmKV);
    prefetch_tmap(&tmO);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < QS; ++s) {
      mbar_init(q_full(s), 1);
      mbar_init(q_empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(k_full(s), 1);
      mbar_init(v_full(s), 1);
      mbar_init(k_empty(s), nqt);                      // one arrival per q tile of the (image, head): the
      mbar_init(v_empty(s), nqt);                      // two issuers release a K/V entry independently
      mbar_init(s_ready(s), 1);
      for (int g = 0; g < 4; ++g) mbar_init(p_part(s, g), 4);
      mbar_init(o_ready(s), 1);
    }
    mbar_init(o_free, 4);
    for (int q = 0; q < 4; ++q) mbar_init(xu_done(q), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<1>(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_launch_dependents();
  pdl_wait();                // the to_qkv GEMM has completed

  // K and V of one (image, head) are loaded once and shared by its q tiles: entry e of the K/V ring
  // belongs to the e-th distinct (image, head) this CTA touches.
  const int bh0 = int(first / nqt);
  if (warp == 0) {
    // ===================== TMA producer =====================
    // Loads are issued in the order they are needed (K, Q, V of an item); every ring slot it
    // waits for was released at least one item ago, so the producer runs well ahead.
    if (elect_one()) {
      for (int i = 0; i < n; ++i) {
        const int64_t item = first + i;
        const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
        const int b = bh / heads, h = bh - b * heads;
        const int e = bh - bh0, es = e & 1;
        const uint32_t eph = (e >> 1) & 1;
        const bool first_of_bh = (i == 0) || (qt == 0);
        if (first_of_bh) {
          mbar_wait(k_empty(es), eph ^ 1u);
          mbar_arrive_expect_tx(k_full(es), L::KV_BYTES);
          tma_load_3d(sK + es * L::KV_BYTES, &tmKV, k_full(es), inner + h * DH, 0, b);
        }
        const int qs = i & (QS - 1);
        mbar_wait(q_empty(qs), ((i / QS) & 1) ^ 1u);
        TRACE(0, i);
        mbar_arrive_expect_tx(q_full(qs), Q_BYTES);
        tma_load_3d(sQ + qs * Q_BYTES, &tmQ, q_full(qs), h * DH, qt * QT, b);
        if (first_of_bh) {
          mbar_wait(v_empty(es), eph ^ 1u);
          TRACE(1, i);
          mbar_arrive_expect_tx(v_full(es), L::KV_BYTES);
          tma_load_3d(sV + es * L::KV_BYTES, &tmKV, v_full(es), 2 * inner + h * DH, 0, b);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 3) {
    // ===================== MMA issuers: warp 1 drives TMEM slot 0, warp 3 slot 1 =====================
    // A slot runs S(i) -> PV(i) -> S(i+2) -> ...  S(i+2) may follow PV(i) at once: one thread's MMAs
    // execute in order, so PV(i) has consumed P(i) before S(i+2) overwrites it, and O has its own
    // columns.  The O accumulator is shared by both slots: PV(i) waits until the epilogue of item
    // i-1 has pulled its O into registers (o_free), which also orders the two issuers' products.
    // Every wait is a blocking mbarrier wait (hardware suspend): no polling next to the softmax warps.
    if (elect_one()) {
      constexpr int fmt = kDT == DT_F16 ? 0 : 1;
      constexpr uint32_t idesc_s = umma_idesc_16(QT, KP, fmt, 0);   // B = K, K-major
      constexpr uint32_t idesc_o = umma_idesc_16(QT, DH, fmt, 1);   // B = V, MN-major
      constexpr int NPARTS = KP >= 128 ? KP / 64 : 1;               // parts of 64 keys (the last takes the remainder)
      const int s = warp == 1 ? 0 : 1;
      const uint32_t d_s = tmem_base + s * SLOT_COLS, d_o = tmem_base + O_COL;
      const int first_lo = int(first % nqt);             // q tile of item 0
      // K/V ring entry of item i.  Every item arrives once on k_empty / v_empty of its entry (the
      // entry is free when all nqt tiles of the (image, head) have); `missing` = tiles of the first
      // (image, head) that belong to the previous CTA, whose arrivals item 0 supplies.
      auto meta = [&](int i, int& es, uint32_t& eph, int& missing) {
        const int t = first_lo + i;                      // tiles since the start of (image, head) bh0
        const int e = t / nqt;
        es = e & 1;
        eph = (e >> 1) & 1;
        missing = i == 0 ? first_lo : 0;
      };
      auto issue_s = [&](int i) {
        int es, missing; uint32_t eph;
        meta(i, es, eph, missing);
        const int qs = i & (QS - 1);
        mbar_wait(q_full(qs), (i / QS) & 1);
        mbar_wait(k_full(es), eph);
        TRACE(2, i);
        tc_fence_after();
        const uint32_t q0 = sQ + qs * Q_BYTES, k0 = sK + es * L::KV_BYTES;
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          umma_bf16_ss<1>(d_s, umma_desc_k_sw128(q0 + k * 32), umma_desc_k_sw128(k0 + k * 32), idesc_s,
                          k != 0 ? 1u : 0u);
        umma_commit(q_empty(qs));
        umma_commit(k_empty(es));
        for (int j = 0; j < missing; ++j) mbar_arrive(k_empty(es));
        umma_commit(s_ready(s));
      };
      if (s < n) issue_s(s);
      for (int i = s; i < n; i += 2) {
        int es, missing; uint32_t eph;
        meta(i, es, eph, missing);
        const uint32_t ph = (i >> 1) & 1;
        const uint32_t v0 = sV + es * L::KV_BYTES;
        // O = P V in parts of 64 keys, each issued as soon as the softmax group has published it
#pragma unroll
        for (int g = 0; g < NPARTS; ++g) {
          mbar_wait(p_part(s, g), ph);
          if (g == 0) {
            mbar_wait(v_full(es), eph);
            mbar_wait(o_free, uint32_t(i & 1) ^ 1u);
            TRACE(3, i);
          }
          tc_fence_after();
          constexpr int KSTEPS = KP / 16;
          const int k_end = g == NPARTS - 1 ? KSTEPS : 4 * g + 4;
#pragma unroll
          for (int kk = 4 * g; kk < k_end; ++kk)
            umma_bf16_ts(d_o, d_s + kk * 8, umma_desc_mn_sw128(v0 + kk * 2048), idesc_o, kk != 0 ? 1u : 0u);
        }
        umma_commit(v_empty(es));
        for (int j = 0; j < missing; ++j) mbar_arrive(v_empty(es));
        umma_commit(o_ready(s));
        if (i + 2 < n) issue_s(i + 2);
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 12) {
    // ===================== softmax (two independent groups) =====================
    const int w = warp - 4;
    const int q = w & 3;                  // TMEM lane quarter (== warp % 4)
    const int grp = w >> 2;               // group == TMEM slot == smem stage parity
    const int row = q * 32 + lane;        // query row in the tile == TMEM lane
    const uint32_t t_slot = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(grp * SLOT_COLS);
    const float sl2 = 0.125f * 1.4426950408889634f;   // dim_head^-0.5 * log2(e)   (vit.py:66)
    // score row = NFULL chunks of 32 columns (+ one of 16); chunks past KMIN may hold keys >= T
    constexpr int NFULL = KP / 32, TAIL = KP % 32;
    constexpr int KMIN = KP == 208 ? 128 : (KP == 128 ? 64 : 0);   // launch_poly: T > KMIN
    static_assert(TAIL == 0 || TAIL == 16, "key block = n*32 (+16)");
    constexpr int NPARTS = KP >= 128 ? KP / 64 : 1;       // P is published in parts of 2 chunks = 64 keys (issuer: same constant)
    static_assert(NPARTS <= 4 && 2 * NPARTS <= NFULL, "parts are pairs of 32-key chunks");

    for (int i = grp; i < n; i += 2) {
      const uint32_t ph = (i >> 1) & 1;
      const int64_t item = first + i;
      const int bh = int(item / nqt), qt = int(item - int64_t(bh) * nqt);
      const bool active = qt * QT + q * 32 < T;          // warp-uniform: any valid query row here?
      if (q == 0 && lane == 0) TRACE(4, i);
      mbar_wait(s_ready(grp), ph);
      if (q == 0 && lane == 0) TRACE(5, i);
      tc_fence_after();
      if (active) {
        // Both passes stream the row through two register buffers: the tcgen05.ld of chunk c+1
        // is in flight while chunk c is processed (tcgen05.wait::ld covers all outstanding loads).
        uint32_t r[2][32];
        // ---- pass 1: row max ----
        float mx = -INFINITY;
        tmem_ld_32x32b_x32p(t_slot, r[0]);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < NFULL; ++c) {
          if (c + 1 < NFULL) tmem_ld_32x32b_x32p(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
          else if (TAIL) tmem_ld_32x32b_x16(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
          uint32_t* rc = r[c & 1];
          if (c * 32 + 32 > KMIN && c * 32 + 32 > T) {   // warp-uniform: only the chunk(s) past T pay
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c * 32 + j >= T) rc[j] = __float_as_uint(-INFINITY);
          }
#pragma unroll
          for (int j = 0; j < 32; j += 2)
            mx = fmaxf(mx, fmaxf(__uint_as_float(rc[j]), __uint_as_float(rc[j + 1])));
          if (c + 1 < NFULL || TAIL) tmem_ld_wait();
        }
        if constexpr (TAIL != 0) {
          uint32_t* rc = r[NFULL & 1];
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (NFULL * 32 + j >= T) rc[j] = __float_as_uint(-INFINITY);
#pragma unroll
          for (int j = 0; j < 16; j += 2)
            mx = fmaxf(mx, fmaxf(__uint_as_float(rc[j]), __uint_as_float(rc[j + 1])));
        }
        if (q == 0 && lane == 0) TRACE(6, i);
        // ---- pass 2: p = exp2((s - max) * scale * log2e), un-normalised; row sum in fp32; P -> TMEM
        // P chunk c (16 columns of 16-bit pairs) lands on S columns [16c, 16c+16), all read already.
        const float mneg = -mx * sl2;
        const unsigned long long sl2x2 = pack_f32x2(sl2, sl2), mnegx2 = pack_f32x2(mneg, mneg);
        unsigned long long la = pack_f32x2(0.f, 0.f), lb = la;
        tmem_ld_32x32b_x32p(t_slot, r[0]);               // the first chunk is in registers before the turn begins
        tmem_ld_wait();
        // The exponential phases of consecutive items take turns on the MUFU of each SMSP (this warp and warp q of
        // the other group share a scheduler): left alone the two groups fall into step (both exponentiate, then both
        // wait), which idles the pipe that bounds this kernel for the length of everything else.
        if (turns) mbar_wait(xu_done(q), uint32_t(i & 1) ^ 1u);
        if (q == 0 && lane == 0) TRACE(9, i);
#pragma unroll
        for (int c = 0; c < NFULL; ++c) {
          if (c + 1 < NFULL) tmem_ld_32x32b_x32p(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
          else if (TAIL) tmem_ld_32x32b_x16(t_slot + (c + 1) * 32, r[(c + 1) & 1]);
          uint32_t pp[16];
          if (c * 32 + 32 > KMIN && c * 32 + 32 > T) softmax_chunk<kDT, 32, true>(r[c & 1], pp, c * 32, T, sl2x2, mnegx2, la, lb);
          else softmax_chunk<kDT, 32, false>(r[c & 1], pp, c * 32, T, sl2x2, mnegx2, la, lb);
          if (c + 1 < NFULL || TAIL) tmem_ld_wait();    // chunk c+1 is in registers: its S columns may go
          if (c >= 2 && (c & 1) == 0 && c / 2 - 1 < NPARTS - 1) {
            // publish part c/2 - 1 (chunks c-2, c-1): their stores were issued a chunk of exponentials ago, so the
            // wait does not stall; the issuer starts that part of P V while this row goes on
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_part(grp, c / 2 - 1));
          }
          tmem_st_32x32b_x16(t_slot + c * 16, pp);
          if (c + 1 == turns) { __syncwarp(); if (lane == 0) mbar_arrive(xu_done(q)); }   // the other group's warp on this SMSP may start
        }
        if constexpr (TAIL != 0) {
          uint32_t pp[8];
          softmax_chunk<kDT, 16, true>(r[NFULL & 1], pp, NFULL * 32, T, sl2x2, mnegx2, la, lb);
          tmem_st_32x32b_x8(t_slot + NFULL * 16, pp);
        }
        if (turns > NFULL) { __syncwarp(); if (lane == 0) mbar_arrive(xu_done(q)); }   // strict alternation
        if (q == 0 && lane == 0) TRACE(11, i);
        float l0, l1;
        unpack_f32x2(add_f32x2(la, lb), l0, l1);
        inv_sh[(i & 3) * 128 + row] = 1.0f / (l0 + l1);   // for the epilogue warps (ordered by the last p_part)
        // training: the row's log-sum-exp in the log2 domain, lse2 = log2 sum_j exp2(s_ij sl2), which lets the adjoint
        // (attention_bwd_tc5.cu) rebuild P block by block without a row maximum
        if (lse_out != nullptr && qt * QT + row < T) lse_out[int64_t(bh) * T + qt * QT + row] = __log2f(l0 + l1) - mneg;
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_part(grp, NPARTS - 1));   // the last part: chunks 2 (NPARTS - 1) .. and the tail
      } else {
        // no valid query row in this warp (last quarter of the 69-row tail tile): keep the hand-offs moving
        if (turns) {
          mbar_wait(xu_done(q), uint32_t(i & 1) ^ 1u);
          if (lane == 0) mbar_arrive(xu_done(q));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int g = 0; g < NPARTS; ++g) mbar_arrive(p_part(grp, g));
        }
      }
      if (q == 0 && lane == 0) TRACE(7, i);
    }
  } else if (warp >= 12) {
    // ===================== epilogue: O / rowsum -> 16-bit -> swizzled smem -> TMA store ==========
    const int q = warp & 3;               // TMEM lane quarter (== warp % 4)
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
      if (leader) TRACE(8, i);
      mbar_wait(o_ready(s), ph);                         // PV(i) done; its last part was issued after p_part(i),
                                                         // which ordered the group's 1/rowsum writes
      tc_fence_after();
      uint32_t o[64];
      float inv = 0.f;
      if (active) {
        tmem_ld_32x32b_x32p(t_lane + O_COL, o);
        tmem_ld_32x32b_x32p(t_lane + O_COL + 32, o + 32);
        inv = inv_sh[(i & 3) * 128 + row];
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free);                // O is in registers: PV(i+1) may overwrite it
      if (active) {
#pragma unroll
        for (int g = 0; g < 8; ++g) {        // 8 columns -> one 16-byte chunk
          st_shared_v4(sOi + uint32_t(row) * 128u + (uint32_t(g ^ (row & 7)) << 4),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 0]) * inv, __uint_as_float(o[g * 8 + 1]) * inv),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 2]) * inv, __uint_as_float(o[g * 8 + 3]) * inv),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 4]) * inv, __uint_as_float(o[g * 8 + 5]) * inv),
                       pack2<kDT>(__uint_as_float(o[g * 8 + 6]) * inv, __uint_as_float(o[g * 8 + 7]) * inv));
        }
      }
      fence_proxy_async_smem();
      // the store of item i-1 (other staging buffer) has been read out: after the barrier every
      // epilogue thread may write that buffer for item i+1
      if (leader) tma_store_wait_read<0>();
      named_bar_sync(1, 128);
      if (leader) {
        tma_store_3d(&tmO, sOi, h * DH, qt * QT, b);     // rows >= T are clipped by the tensor map
        tma_store_commit();
        TRACE(10, i);
      }
    }
    if (leader) tma_store_wait<0>();                     // smem must outlive the last bulk store
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

// How the two softmax groups share the XU of each SMSP (VITB200_ATTN_TURNS): 0 = free-running; h in 1..6 = a warp lets
// its partner (warp q of the other group, next item) start pass 2 once it has finished its own chunk h - 1 of 32 keys,
// so the two exponential phases overlap from there on; 7 = strict alternation (hand-off after the last exponential).
// Measured at ViT-B/16 batch 256 (profiles/r02_attention.md): 0..3 85-86 us, 4 and 5 84 us, 6 and 7 95 us; the default
// is the chunk before the last full one (5 at 208 keys).
int attn_turns() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VITB200_ATTN_TURNS");
    v = (e && e[0] >= '0' && e[0] <= '9') ? e[0] - '0' : -1;   // default: hand-off one chunk before the last
  }
  return v;
}

template <int kDT, int KP>
int launch_kp(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads, float* lse, int q_tiles) {
  using L = Smem<KP>;
  static PerDevice<bool> configured_on;   // the smem opt-in is per (function, device)
  if (bool& configured = configured_on.here(); !configured) {
    VB_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<kDT, KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    configured = true;
  }
  const int inner = heads * DH;
  CUtensorMap tq, tkv, to;
  int rc;
  if ((rc = make_tmap_3d_16(&tq, qkv, batch, T, 3 * inner, 3 * inner, QT, kDT))) return rc;
  if ((rc = make_tmap_3d_16(&tkv, qkv, batch, T, 3 * inner, 3 * inner, KP, kDT))) return rc;
  if ((rc = make_tmap_3d_16(&to, out, batch, T, inner, inner, QT, kDT))) return rc;
  // items are (image, head, q tile) with nqt q tiles per (image, head): fewer than ceil(T / QT) computes only the first
  // query rows of every image (the class-token tail of the forward needs q tile 0 alone)
  const int nqt = q_tiles > 0 && q_tiles < ceil_div(T, QT) ? q_tiles : ceil_div(T, QT);
  const int64_t items64 = int64_t(batch) * heads * nqt;
  if (items64 > 0x7fffffff) return fail(VITB200_ERR_INVALID, "attention: too many work items");
  const int items = int(items64);
  const int grid = items < sm_count() ? items : sm_count();
  VB_CUDA(launch_kernel(attention_tc5_kernel<kDT, KP>, dim3(grid), dim3(NT), L::TOTAL, stream, 1,
                        tq, tkv, to, T, heads, nqt, items, attn_turns(), lse));
  VB_LAUNCH_CHECK("attention_tc5_kernel");
  return 0;
}

template <int kDT>
int launch_dt(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads, float* lse, int q_tiles) {
  if (T <= 64) return launch_kp<kDT, 64>(stream, qkv, out, batch, T, heads, lse, q_tiles);      // KMIN: T > 0 / 64 / 128
  if (T <= 128) return launch_kp<kDT, 128>(stream, qkv, out, batch, T, heads, lse, q_tiles);
  return launch_kp<kDT, 208>(stream, qkv, out, batch, T, heads, lse, q_tiles);
}

}  // namespace

#ifdef VITB200_TRACE
}  // namespace vb
extern "C" int vitb200_debug_attention_trace(long long* host, int n) {
  return cudaMemcpyFromSymbol(host, vb::g_trace, sizeof(long long) * (n < 12 * 64 ? n : 12 * 64)) == cudaSuccess ? 0 : -2;
}
namespace vb {
#endif

bool attention_tc5_supports(int T) { return T >= 1 && T <= 208; }

int launch_attention_tc5(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads,
                         int dtype, float* lse, int q_tiles) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention: empty problem");
  if (!attention_tc5_supports(T)) return fail(VITB200_ERR_UNSUPPORTED, "attention_tc5: T > 208");
  if (dtype == DT_BF16) return launch_dt<DT_BF16>(stream, qkv, out, batch, T, heads, lse, q_tiles);
  if (dtype == DT_F16) return launch_dt<DT_F16>(stream, qkv, out, batch, T, heads, lse, q_tiles);
  return fail(VITB200_ERR_INVALID, "attention: dtype must be bf16 or fp16");
}

}  // namespace vb
