// ptx.cuh -- thin inline-PTX wrappers for sm_100a: mbarrier, TMA, tcgen05/TMEM, elect.sync.
// No CUTLASS/CuTe dependency.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

namespace vb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
// One lane of a CONVERGED warp.  Unlike `lane == 0`, the compiler knows that exactly one lane is inside the branch: single-
// thread instructions (tcgen05.mma / commit, TMA) are emitted as they are, on the uniform datapath, instead of each inside an
// ELECT / PLOP3 / BRA.U.ANY loop over the possibly-active lanes (7 instead of 10-16 SASS instructions per tcgen05.mma, and the
// issuing thread is latency-bound on exactly that chain: profiles/r02_attention_bwd.md).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------- programmatic dependent launch
// Every kernel of the forward is launched with programmatic stream serialization: its CTAs may
// start (barrier init, TMEM allocation, descriptor prefetch) while the previous kernel drains, and
// pdl_wait() holds them until that kernel has completed and its writes are visible.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
// Arrive on the barrier at the same smem offset in CTA `cta` of the cluster.  RELAXED: callers
// order their own side first (tcgen05.wait::ld + tcgen05.fence::before_thread_sync); a
// cluster-scope release here stalls the warp for >1000 cycles.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(cta) : "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `cta` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
  return r;
}
// arrive on a barrier given by its shared::cluster address
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// non-blocking probe (no hardware suspend): for a thread that polls several barriers
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// Spin with a watchdog: a protocol bug traps (launch fails with an error) instead of
// hanging the GPU.  ~4e9 cycles is seconds, far beyond any legitimate wait here.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      if ((threadIdx.x & 31) == 0)   // one line per warp: the set of stuck waits is the diagnosis
        printf("vitb200: mbarrier wait timed out (block %d warp %d bar 0x%x parity %u)\n",
               int(blockIdx.x), int(threadIdx.x >> 5), bar, parity);
      __trap();
    }
  }
}
// cluster-scope acquire wait (barrier completed by a remote CTA's arrive)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (!ok && clock64() - t0 > 4000000000LL) {
      printf("vitb200: cluster mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n",
             int(blockIdx.x), int(threadIdx.x), bar, parity);
      __trap();
    }
  }
}

// ----------------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, uint32_t bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// 2-CTA flavour: the transaction bytes land on the barrier address given (the
// caller passes the leader CTA's barrier, i.e. its shared::cluster address).
__device__ __forceinline__ void tma_load_2d_cg2(uint32_t dst, const void* tmap, uint32_t bar,
                                                int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// multicast flavour: the box lands at the same smem offset of every CTA in `cta_mask`, and each
// destination signals the barrier at `bar`'s offset in its own pair leader
__device__ __forceinline__ void tma_load_2d_cg2_mc(uint32_t dst, const void* tmap, uint32_t bar,
                                                   int32_t c0, int32_t c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}

// TMA stores (smem -> global), bulk-group completion.  OOB parts of the box are clipped.
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
// global[tile] += smem[tile] performed by the memory system (element type from the tensor map)
__device__ __forceinline__ void tma_reduce_add_2d(const void* tmap, uint32_t src, int32_t c0, int32_t c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const void* tmap, uint32_t src, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* tmap, uint32_t bar,
                                            int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// im2col-mode load of an NDHWC tensor (cuTensorMapEncodeIm2col, rank 5): `pixelsPerColumn` output pixels starting at base
// pixel (w, h, d, n), walked along W, then H, then D, then N inside the map's bounding box of filter origins,
// `channelsPerPixel` channels from c each; the filter tap (w_off, h_off, d_off) is added to every pixel.  Lands as a dense
// [pixels, channels] tile.
__device__ __forceinline__ void tma_load_im2col_5d(uint32_t dst, const void* tmap, uint32_t bar, int32_t c, int32_t w,
                                                   int32_t h, int32_t d, int32_t n, uint16_t w_off, uint16_t h_off,
                                                   uint16_t d_off) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2], {%8, %9, %10};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(d), "r"(n), "h"(w_off),
        "h"(h_off), "h"(d_off)
      : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {   // <= N groups may still be reading smem
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {        // <= N groups not yet complete
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float4 ld_shared_v4f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ------------------------------------------------------------ tcgen05 / TMEM
template <int kCtaGroup>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  if constexpr (kCtaGroup == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]; single thread issues.
template <int kCtaGroup>
__device__ __forceinline__ void umma_bf16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  }
}
// The same with 8-bit floating-point operands (kind::f8f6f4: K = 32 per instruction, still 32 bytes of a 128-byte row)
template <int kCtaGroup>
__device__ __forceinline__ void umma_f8_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                           uint32_t idesc, uint32_t accumulate) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  }
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// make `bar` complete once all previously issued tcgen05.mma of this thread retire
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
               ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit_cg2_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64"
      " [%0], %1;" ::"r"(bar), "h"(cta_mask) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane
// (taddr.lane + i), registers r[0..31] = columns taddr.col + 0..31.
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7])
      : "r"(taddr) : "memory");
}
// pointer flavour of the x32 load (register array slices)
__device__ __forceinline__ void tmem_ld_32x32b_x32p(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]),
        "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]),
        "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]),
        "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x4(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor, K-major operand, SWIZZLE_128B, rows of 128 B
// (64 bf16), 8-row groups 1024 B apart.  `addr` must lie in a 1024 B-aligned
// tile; advancing K by 16 bf16 inside the 128 B row = +32 B on the address.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t addr) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4)      // start address  [0,14)
         | (1ull << 16)                                      // LBO (unused for swizzled K-major)
         | (64ull << 32)                                     // SBO = 1024 B >> 4  [32,46)
         | (1ull << 46)                                      // descriptor version (Blackwell)
         | (2ull << 61);                                     // SWIZZLE_128B
}
// MN-major operand, SWIZZLE_128B: 64 MN-elements (128 B) contiguous per K row,
// 8 K-rows per 1024 B group (SBO); one atom wide along MN so LBO is unused.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t addr) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) |
         (1ull << 46) | (2ull << 61);
}
// The same for an operand several 64-element atoms wide along MN: atom j starts `lbo_bytes` after
// atom j-1 (canonical layout ((8,8,m),(8,k)) : ((1,8,LBO),(64,SBO)) in 16-bit elements).
__device__ __forceinline__ uint64_t umma_desc_mn_sw128_wide(uint32_t addr, uint32_t lbo_bytes) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>(lbo_bytes >> 4) << 16) |
         (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// The same descriptors split into words, for issue loops that walk an operand by a constant stride: only the low
// word changes (start address >> 4 in bits [0,14), LBO >> 4 in [16,30)), so the k-th descriptor is `lo + k * (stride >> 4)`
// -- one uniform add per operand in front of the tcgen05.mma instead of the shift / mask / or chain (the issuing thread
// pays for every instruction of that chain: profiles/microbench/mma_chain.cu, profiles/r02_attention_bwd.md).
constexpr uint32_t UMMA_DESC_HI_SW128 = 0x40004040u;   // SBO 1024 B, version 1, SWIZZLE_128B
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t addr, uint32_t lbo_bytes = 16) {
  return ((addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16);
}
// D[tmem] (+)= A * B, both from shared memory, descriptors given by their low words (SWIZZLE_128B, cta_group::1)
__device__ __forceinline__ void umma_bf16_ss_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(UMMA_DESC_HI_SW128) : "memory");
}

// kind::f16 instruction descriptor: (bf16 | fp16) x same -> fp32; operand majors selectable.
// `fmt`: 0 = F16, 1 = BF16 (UMMA F16F32Format).
__host__ __device__ constexpr uint32_t umma_idesc_16(int M, int N, int fmt, int b_mn_major = 0, int a_mn_major = 0) {
  return (1u << 4)                       // D format  : F32
         | (uint32_t(fmt) << 7)          // A format
         | (uint32_t(fmt) << 10)         // B format
         | (uint32_t(a_mn_major) << 15)  // A major   : 0 = K, 1 = MN
         | (uint32_t(b_mn_major) << 16)  // B major   : 0 = K, 1 = MN
         | (uint32_t(N >> 3) << 17)      // N >> 3
         | (uint32_t(M >> 4) << 24);     // M >> 4
}
// kind::f8f6f4 instruction descriptor, both operands E4M3 and K-major, D fp32.  The PTX ISA's table for .kind::f8f6f4
// puts the A / B formats in bits [7,10) / [10,13) with E4M3 = 0, E5M2 = 1, E2M3 = 3, E3M2 = 4, E2M1 = 5; the other
// fields sit where they do for kind::f16.
__host__ __device__ constexpr uint32_t umma_idesc_e4m3(int M, int N) {
  return (1u << 4)                       // D format  : F32
         | (0u << 7)                     // A format  : E4M3
         | (0u << 10)                    // B format  : E4M3
         | (uint32_t(N >> 3) << 17)      // N >> 3
         | (uint32_t(M >> 4) << 24);     // M >> 4
}

// ------------------------------------------------------------------- cluster
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 16-bit storage formats of the tensor-core path (values of VITB200_DT_*)
constexpr int DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2;
constexpr int DT_E4M3 = 3;   // 8-bit E4M3 operands of the fp8 precision (1 byte per element)

// four fp32 -> four E4M3 codes (round to nearest even, saturated to +-448), v0 in bits [0,8)
__device__ __forceinline__ uint32_t pack4_e4m3(float v0, float v1, float v2, float v3) {
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(v1), "f"(v0));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(v3), "f"(v2));
  return uint32_t(lo) | (uint32_t(hi) << 16);
}

// two fp32 -> packed 16-bit pair (lo in bits [0,16)); fp16 saturates to +-65504 instead of inf
template <int kDT>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t r;
  if constexpr (kDT == DT_F16) {
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  } else {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  }
  return r;
}
template <int kDT>
__device__ __forceinline__ uint16_t cvt16(float v) {
  return static_cast<uint16_t>(pack2<kDT>(v, 0.f) & 0xFFFFu);
}
template <int kDT>
__device__ __forceinline__ float to_f32(uint16_t h) {
  if constexpr (kDT == DT_F16) return __half2float(__ushort_as_half(h));
  else return __uint_as_float(uint32_t(h) << 16);
}
// packed fp32x2 arithmetic (sm_100): one issue slot for two lanes of FFMA / FADD
__device__ __forceinline__ unsigned long long pack_f32x2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma_f32x2(unsigned long long a, unsigned long long b,
                                                        unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ unsigned long long mul_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ unsigned long long add_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// ------------------------------------------------------------------- dropout
// nn.Dropout(rate)(x, deterministic=False) (vit.py:50,52,83,155): keep with probability 1 - rate,
// scale kept values by 1 / (1 - rate).  Counter-based Philox4x32-10 keyed by the 'dropout' rng the
// caller passes: the mask of element e of dropout site s is a pure function of (key, s, e), like
// Flax's functional rng -- same key, same mask.  (Bit parity with JAX's threefry is impossible
// without JAX; oracle/philox.py restates this generator so the tests inject identical masks.)
struct Dropout {
  uint32_t key_lo = 0, key_hi = 0;   // 'dropout' rng key
  uint32_t site = 0;                 // which nn.Dropout instance (0 = emb, 1+3l.. per layer)
  uint32_t threshold = 0;            // drop when rand32 < threshold; 0 = rate 0 = off
  float inv_keep = 1.f;
};
// four 32-bit random words for elements [4*quad, 4*quad+4) of the site
__device__ __forceinline__ uint4 philox4x32_10(unsigned long long quad, uint32_t site, uint32_t k0, uint32_t k1) {
  uint32_t c0 = uint32_t(quad), c1 = uint32_t(quad >> 32), c2 = site, c3 = 0u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
// apply the site's mask to 4 consecutive elements starting at flat index `elem` (a multiple of 4)
__device__ __forceinline__ void dropout4(const Dropout& d, long long elem, float& a, float& b, float& c, float& e) {
  const uint4 r = philox4x32_10(static_cast<unsigned long long>(elem) >> 2, d.site, d.key_lo, d.key_hi);
  a = r.x < d.threshold ? 0.f : a * d.inv_keep;
  b = r.y < d.threshold ? 0.f : b * d.inv_keep;
  c = r.z < d.threshold ? 0.f : c * d.inv_keep;
  e = r.w < d.threshold ? 0.f : e * d.inv_keep;
}

// LayerNorm folded into the GEMMs around it (gemm_tc.cu header).  Producers (RESID_LN, TOKENS_LN) write `x16`
// ([M, N] 16-bit copy of their fp32 output) and `stats` ([M, slots] partial (sum, sum of squares) of each output row,
// slot = 2 * n_tile + epilogue group); consumers (LN_STORE_16, LN_GELU_16) read `stats` of their A rows and `c`.
struct LnFold {
  void* x16 = nullptr;
  float2* stats = nullptr;
  const float* c = nullptr;
  int slots = 0;
  float eps = 1e-6f;
};

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

}  // namespace vb
