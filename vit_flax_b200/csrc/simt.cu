// simt.cu -- the CUDA-core kernels of the path:
//   K2  LayerNorm (warp-shuffle, vectorised; fp32 in, 16-bit or fp32 out)    vit.py:31,163
//   K1a patchify + fp32->16-bit cast (im2col folded into the mandatory cast) vit.py:146
//       and its adjoint, unpatchify (fp32 patch-feature gradient -> image gradient)
//   K1b cls rows (fp32 mode; the tensor-core path writes them in the patch GEMM) vit.py:151-153
//   K5a pool (cls / mean) + head LayerNorm                                   vit.py:159-163
//   K7  weight pack (fp32 [K,N] -> 16-bit [N,Kpad])
//   fp32 validation mode: SIMT GEMM with the same fused epilogues and a
//   straightforward fp32 attention (tolerance 1e-4 against the oracle).
#include <cstdlib>

#include "common.h"
#include "ptx.cuh"

namespace vb {

namespace {

// eps is a kernel argument: 1e-6 = flax nn.LayerNorm default (vit.py:31,163; NOT torch's 1e-5),
// 1e-5 for SimpleViT's LayerNorm(epsilon = 1e-5) (simple_vit.py:41,58,118)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------- LayerNorm (K2)
// One warp per row, the row lives in registers (<= 16 float4 per lane => dim <= 2048).
template <int NV, int kDT, bool kCopy>
__global__ void __launch_bounds__(256)
layernorm_rows_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                      const float* __restrict__ bias, void* __restrict__ y, int rows, int dim, int reverse, float eps,
                      float* __restrict__ copy,     // copy != null (training): also x -> copy, the next residual buffer
                      int64_t ldx) {                // row pitch of x (y and copy are dense)
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Rows are walked from the END of the residual stream: the GEMM that just updated x wrote its
  // last row blocks last, so they are what the 126 MB L2 still holds of the 155 MB stream, and the
  // GEMM that follows starts with the row blocks this kernel wrote last (VITB200_LN_REVERSE=0: off).
  const int row = reverse ? rows - 1 - (blockIdx.x * 8 + warp) : blockIdx.x * 8 + warp;
  if (row < 0 || row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + int64_t(row) * ldx);
  const int nvec = dim >> 2;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 32 + lane;
    if (c < nvec) {
      v[i] = __ldcs(xr + c);
      if constexpr (kCopy) reinterpret_cast<float4*>(copy + int64_t(row) * dim)[c] = v[i];
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    } else {
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const float mean = warp_sum(s) / float(dim);
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 32 + lane;
    if (c < nvec) {
      const float a = v[i].x - mean, b = v[i].y - mean, cc = v[i].z - mean, d = v[i].w - mean;
      ss += (a * a + b * b) + (cc * cc + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(ss) / float(dim) + eps);
  const float4* g4 = reinterpret_cast<const float4*>(scale);
  const float4* b4 = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 32 + lane;
    if (c < nvec) {
      const float4 g = __ldg(g4 + c), b = __ldg(b4 + c);
      float4 o;
      o.x = (v[i].x - mean) * rstd * g.x + b.x;
      o.y = (v[i].y - mean) * rstd * g.y + b.y;
      o.z = (v[i].z - mean) * rstd * g.z + b.z;
      o.w = (v[i].w - mean) * rstd * g.w + b.w;
      if constexpr (kDT == DT_E4M3) {   // the A operand of the fp8 GEMMs: normalised, unscaled, saturated
        reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(y) + int64_t(row) * dim)[c] = pack4_e4m3(o.x, o.y, o.z, o.w);
      } else if constexpr (kDT != DT_F32) {
        uint2 p;
        p.x = pack2<kDT>(o.x, o.y);
        p.y = pack2<kDT>(o.z, o.w);
        reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(y) + int64_t(row) * dim)[c] = p;
      } else {
        reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + int64_t(row) * dim)[c] = o;
      }
    }
  }
}

// Any dim: one warp per row, three passes over the (cached) row.
template <int kDT>
__global__ void __launch_bounds__(256)
layernorm_generic_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                         const float* __restrict__ bias, void* __restrict__ y, int rows, int dim, float eps, int64_t ldx) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const float* xr = x + int64_t(row) * ldx;
  float s = 0.f;
  for (int c = lane; c < dim; c += 32) s += xr[c];
  const float mean = warp_sum(s) / float(dim);
  float ss = 0.f;
  for (int c = lane; c < dim; c += 32) { const float d = xr[c] - mean; ss += d * d; }
  const float rstd = rsqrtf(warp_sum(ss) / float(dim) + eps);
  for (int c = lane; c < dim; c += 32) {
    const float o = (xr[c] - mean) * rstd * scale[c] + bias[c];
    if constexpr (kDT == DT_E4M3) reinterpret_cast<uint8_t*>(y)[int64_t(row) * dim + c] = uint8_t(pack4_e4m3(o, 0.f, 0.f, 0.f) & 0xFFu);
    else if constexpr (kDT != DT_F32) reinterpret_cast<uint16_t*>(y)[int64_t(row) * dim + c] = cvt16<kDT>(o);
    else reinterpret_cast<float*>(y)[int64_t(row) * dim + c] = o;
  }
}

int ln_reverse() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VITB200_LN_REVERSE");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v;
}

template <int kDT>
int launch_ln_t(cudaStream_t st, const float* x, const float* g, const float* b, void* y, int rows,
                int dim, float eps, float* copy, int64_t ldx) {
  const int grid = ceil_div(rows, 8);
  const bool vec = (dim % 4 == 0) && (ldx % 4 == 0) && dim <= 2048 &&
                   ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) |
                     reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(b)) & 15) == 0;
  if (!vec || (reinterpret_cast<uintptr_t>(copy) & 15) != 0) {
    if (copy != nullptr) VB_CUDA(cudaMemcpyAsync(copy, x, size_t(rows) * dim * sizeof(float), cudaMemcpyDeviceToDevice, st));
    VB_CUDA(launch_kernel(layernorm_generic_kernel<kDT>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, eps, ldx));
  } else {
    const int nv = ceil_div(dim, 128);
    if (nv <= 4) { if (copy) VB_CUDA(launch_kernel(layernorm_rows_kernel<4, kDT, true>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx));
                   else VB_CUDA(launch_kernel(layernorm_rows_kernel<4, kDT, false>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx)); }
    else if (nv <= 6) { if (copy) VB_CUDA(launch_kernel(layernorm_rows_kernel<6, kDT, true>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx));
                        else VB_CUDA(launch_kernel(layernorm_rows_kernel<6, kDT, false>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx)); }
    else if (nv <= 8) { if (copy) VB_CUDA(launch_kernel(layernorm_rows_kernel<8, kDT, true>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx));
                        else VB_CUDA(launch_kernel(layernorm_rows_kernel<8, kDT, false>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx)); }
    else if (nv <= 10) { if (copy) VB_CUDA(launch_kernel(layernorm_rows_kernel<10, kDT, true>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx));
                         else VB_CUDA(launch_kernel(layernorm_rows_kernel<10, kDT, false>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx)); }
    else { if (copy) VB_CUDA(launch_kernel(layernorm_rows_kernel<16, kDT, true>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx));
           else VB_CUDA(launch_kernel(layernorm_rows_kernel<16, kDT, false>, dim3(grid), dim3(256), 0, st, 1, x, g, b, y, rows, dim, ln_reverse(), eps, copy, ldx)); }
  }
  VB_LAUNCH_CHECK("layernorm");
  return 0;
}

// -------------------------------------------------------------- patchify (K1a)
// out[(b*Np + t), f], f = (p1*pw + p2)*C + c  <-  x[b, hh*ph+p1, ww*pw+p2, c]; zero pad f >= K0.
// tok_off = 1 writes the TOKEN layout instead: row b*(Np+1) + 1 + t, leaving row b*(Np+1) (the image's
// class-token slot, never written, never used as data) so that the patch GEMM's output rows are the
// token rows themselves (VITB200_EPI_TOKENS_F32).
template <int kDT>
__global__ void __launch_bounds__(256)
patchify_kernel(const float* __restrict__ img, void* __restrict__ out, int batch, int H, int W,
                int C, int ph, int pw, int Kpad, int nchw, int tok_off) {
  pdl_launch_dependents();
  pdl_wait();
  const int gw = W / pw, gh = H / ph;
  const int K0 = ph * pw * C;
  const int64_t pairs_per_row = Kpad >> 1;     // Kpad is even
  const int64_t total = int64_t(batch) * gh * gw * pairs_per_row;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total;
       i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t prow = i / pairs_per_row;
    const int f0 = int(i - prow * pairs_per_row) * 2;
    const int t = int(prow % (gh * gw));
    const int b = int(prow / (gh * gw));
    const int hh = t / gw, ww = t - hh * gw;
    float v[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int f = f0 + e;
      if (f < K0) {
        const int c = f % C, pp = f / C;
        const int p1 = pp / pw, p2 = pp - p1 * pw;
        // NHWC (vit.py:146) or NCHW (simple_vit.py:125: 'b c (h p1) (w p2) -> b h w (p1 p2 c)')
        v[e] = nchw ? __ldg(img + ((int64_t(b) * C + c) * H + hh * ph + p1) * W + ww * pw + p2)
                    : __ldg(img + ((int64_t(b) * H + hh * ph + p1) * W + ww * pw + p2) * C + c);
      } else {
        v[e] = 0.f;
      }
    }
    // token layout (tok_off = 1): image b's patches start one row late, behind its class-token row
    const int64_t o = i + (int64_t(b) + 1) * tok_off * pairs_per_row;
    if constexpr (kDT != DT_F32) {
      reinterpret_cast<uint32_t*>(out)[o] = pack2<kDT>(v[0], v[1]);
    } else {
      reinterpret_cast<float2*>(out)[o] = make_float2(v[0], v[1]);
    }
  }
}

// Fast path (pw*C even, which covers every config of the path): walk the IMAGE ROWS.  Row (b, y) is
// W*C contiguous floats and is made of gw patch-row segments of pw*C floats; segment ww lands at
// out[(b, hh, ww), p1*pw*C ...] with y = hh*ph + p1.  One float2 per thread: coalesced reads, writes
// in runs of pw*C 16-bit values (96 B at P = 16).  The pad columns K0..Kpad are zeroed by a second
// grid-stride loop, so the buffer needs no memset.
template <int kDT>
__global__ void __launch_bounds__(256)
patchify_rows_kernel(const float* __restrict__ img, void* __restrict__ out, int batch, int H, int W,
                     int C, int ph, int pw, int Kpad, int tok_off) {   // NHWC only; NCHW goes through patchify_kernel
  pdl_launch_dependents();
  pdl_wait();
  const int gw = W / pw, gh = H / ph;
  const int seg = pw * C;                 // floats per patch-row segment (even)
  const int pairs_per_row = (W * C) >> 1;
  const int K0 = ph * seg;
  const int pad_pairs = (Kpad - K0) >> 1;
  const int64_t total = int64_t(batch) * H * pairs_per_row;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = i / pairs_per_row;                 // image row (b, y)
    const int t = int(i - r * pairs_per_row);
    const int b = int(r / H), y = int(r - int64_t(b) * H);
    const int hh = y / ph, p1 = y - hh * ph;
    const float2 v = __ldcs(reinterpret_cast<const float2*>(img) + i);
    const int x = t * 2;
    const int ww = x / seg, rem = x - ww * seg;
    const int64_t o = ((int64_t(b) * gh + hh) * gw + ww + (int64_t(b) + 1) * tok_off) * Kpad + p1 * seg + rem;   // even
    if constexpr (kDT != DT_F32) reinterpret_cast<uint32_t*>(out)[o >> 1] = pack2<kDT>(v.x, v.y);
    else reinterpret_cast<float2*>(out)[o >> 1] = v;
  }
  if (pad_pairs > 0) {
    const int64_t npad = int64_t(batch) * gh * gw * pad_pairs;
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < npad; i += int64_t(gridDim.x) * blockDim.x) {
      const int64_t patch = i / pad_pairs;
      const int k = int(i - patch * pad_pairs);
      const int64_t o = (patch + (patch / (gh * gw) + 1) * tok_off) * Kpad + K0 + 2 * k;
      if constexpr (kDT != DT_F32) reinterpret_cast<uint32_t*>(out)[o >> 1] = 0u;
      else reinterpret_cast<float2*>(out)[o >> 1] = make_float2(0.f, 0.f);
    }
  }
}

// Fastest path (pw*C and W*C multiples of 4, 16-byte aligned images: every /16 and /14 RGB config):
// a block walks IMAGE ROWS (b, y), one float4 per thread and row -- one integer division per float4
// instead of four per element, fully coalesced 16-byte loads, 8-byte stores.
template <int kDT>
__global__ void __launch_bounds__(256)
patchify_row4_kernel(const float* __restrict__ img, void* __restrict__ out, int rows, int H, int W, int C,
                     int ph, int pw, int Kpad, int tok_off) {
  pdl_launch_dependents();
  pdl_wait();
  const int gw = W / pw, gh = H / ph;
  const int seg4 = (pw * C) >> 2;          // float4 per patch-row segment
  const int n4 = (W * C) >> 2;             // float4 per image row
  const int K0 = ph * pw * C;
  const int pad2 = (Kpad - K0) >> 1;
  constexpr int U = 4;                      // image rows in flight per thread (memory-level parallelism)
  for (int r0 = blockIdx.x; r0 < rows; r0 += U * gridDim.x) {   // image row index b*H + y
    for (int t = threadIdx.x; t < n4; t += blockDim.x) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * gridDim.x;
        if (r < rows) v[u] = __ldcs(reinterpret_cast<const float4*>(img + int64_t(r) * W * C) + t);
      }
      const int ww = t / seg4, rem4 = t - ww * seg4;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * gridDim.x;
        if (r >= rows) break;
        const int b = r / H, y = r - b * H;
        const int hh = y / ph, p1 = y - hh * ph;
        const int64_t o = ((int64_t(b) * gh + hh) * gw + ww + (b + 1) * tok_off) * Kpad + p1 * (seg4 << 2) + (rem4 << 2);   // multiple of 4
        if constexpr (kDT != DT_F32) {
          uint2 p;
          p.x = pack2<kDT>(v[u].x, v[u].y);
          p.y = pack2<kDT>(v[u].z, v[u].w);
          reinterpret_cast<uint2*>(out)[o >> 2] = p;
        } else {
          reinterpret_cast<float4*>(out)[o >> 2] = v[u];
        }
      }
    }
    // zero the pad columns K0..Kpad once per patch (by the block that holds the patch's last image row)
    if (pad2 > 0) {
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * gridDim.x;
        if (r >= rows) break;
        const int b = r / H, y = r - b * H;
        const int hh = y / ph, p1 = y - hh * ph;
        if (p1 != ph - 1) continue;
        const int64_t patch0 = (int64_t(b) * gh + hh) * gw + (b + 1) * tok_off;
        for (int t = threadIdx.x; t < gw * pad2; t += blockDim.x) {
          const int ww = t / pad2, k = t - ww * pad2;
          const int64_t o = (patch0 + ww) * Kpad + K0 + 2 * k;
          if constexpr (kDT != DT_F32) reinterpret_cast<uint32_t*>(out)[o >> 1] = 0u;
          else reinterpret_cast<float2*>(out)[o >> 1] = make_float2(0.f, 0.f);
        }
      }
    }
  }
}

// ------------------------------------------------------ unpatchify (adjoint of K1a)
// img[b, y, x, c] (or img[b, c, y, x]) = patches[row(b, patch of (y, x)), f(y, x, c)] -- the transpose of the patchify
// permutation, fp32 in and out.  Patches do not overlap, so every pixel is written exactly once (no accumulation); the
// pad columns K0..Kpad and the class-token slot rows (tok_off = 1) are never read.
__global__ void __launch_bounds__(256)
unpatchify_kernel(const float* __restrict__ patches, float* __restrict__ img, int batch, int H, int W, int C,
                  int ph, int pw, int Kpad, int nchw, int tok_off) {
  pdl_launch_dependents();
  pdl_wait();
  const int gw = W / pw, gh = H / ph;
  const int64_t total = int64_t(batch) * H * W * C;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    int64_t r = i;
    int b, y, x, c;
    if (nchw) {
      x = int(r % W); r /= W;
      y = int(r % H); r /= H;
      c = int(r % C); b = int(r / C);
    } else {
      c = int(r % C); r /= C;
      x = int(r % W); r /= W;
      y = int(r % H); b = int(r / H);
    }
    const int hh = y / ph, p1 = y - hh * ph, ww = x / pw, p2 = x - ww * pw;
    const int64_t row = (int64_t(b) * gh + hh) * gw + ww + (int64_t(b) + 1) * tok_off;
    img[i] = __ldcs(patches + row * Kpad + (p1 * pw + p2) * C + c);
  }
}

// NHWC fast path (pw*C and Kpad multiples of 4, 16-byte aligned buffers), the mirror of patchify_row4_kernel: a block
// walks IMAGE ROWS (b, y); each float4 of the row is one 16-byte piece of a pw*C patch-row segment, read from the patch
// matrix and stored coalesced into the image row.
__global__ void __launch_bounds__(256)
unpatchify_row4_kernel(const float* __restrict__ patches, float* __restrict__ img, int rows, int H, int W, int C,
                       int ph, int pw, int Kpad, int tok_off) {
  pdl_launch_dependents();
  pdl_wait();
  const int gw = W / pw, gh = H / ph;
  const int seg4 = (pw * C) >> 2;          // float4 per patch-row segment
  const int n4 = (W * C) >> 2;             // float4 per image row
  constexpr int U = 4;                      // image rows in flight per thread (memory-level parallelism)
  for (int r0 = blockIdx.x; r0 < rows; r0 += U * gridDim.x) {   // image row index b*H + y
    for (int t = threadIdx.x; t < n4; t += blockDim.x) {
      const int ww = t / seg4, rem4 = t - ww * seg4;
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * gridDim.x;
        if (r < rows) {
          const int b = r / H, y = r - b * H;
          const int hh = y / ph, p1 = y - hh * ph;
          const int64_t o = ((int64_t(b) * gh + hh) * gw + ww + (b + 1) * tok_off) * Kpad + p1 * (seg4 << 2) + (rem4 << 2);
          v[u] = __ldcs(reinterpret_cast<const float4*>(patches + o));
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * gridDim.x;
        if (r < rows) reinterpret_cast<float4*>(img + int64_t(r) * W * C)[t] = v[u];
      }
    }
  }
}

// -------------------------------------------------------------- cls rows (K1b)
__global__ void cls_rows_kernel(const float* __restrict__ cls, const float* __restrict__ pos,
                                float* __restrict__ x, int batch, int T, int dim, Dropout drop) {
  pdl_launch_dependents();
  pdl_wait();
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= int64_t(batch) * dim) return;
  const int b = int(i / dim), d = int(i - int64_t(b) * dim);
  float v = cls[d] + pos[d];
  if (drop.threshold != 0) {   // emb dropout (vit.py:155): same flat index as the patch rows use
    const int64_t e = int64_t(b) * T * dim + d;
    const uint4 r = philox4x32_10(static_cast<unsigned long long>(e) >> 2, drop.site, drop.key_lo, drop.key_hi);
    const uint32_t w = (e & 3) == 0 ? r.x : (e & 3) == 1 ? r.y : (e & 3) == 2 ? r.z : r.w;
    v = w < drop.threshold ? 0.f : v * drop.inv_keep;
  }
  x[int64_t(b) * T * dim + d] = v;
}

// ------------------------------------------------- pool + head LayerNorm (K5a)
template <int kDT>
__global__ void __launch_bounds__(256)
pool_layernorm_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                      const float* __restrict__ bias, void* __restrict__ y, int T, int dim,
                      int pool, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sh[];          // dim floats + 16 reduction slots
  float* pooled = sh;
  float* red = sh + dim;
  const int b = blockIdx.x;
  const float* xb = x + int64_t(b) * T * dim;
  float s = 0.f;
  for (int d = threadIdx.x; d < dim; d += blockDim.x) {
    float v;
    if (pool == VITB200_POOL_MEAN) {
      float acc = 0.f;
      for (int t = 0; t < T; ++t) acc += xb[int64_t(t) * dim + d];
      v = acc / float(T);
    } else {
      v = xb[d];
    }
    pooled[d] = v;
    s += v;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  s = warp_sum(s);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < 8; ++w) tot += red[w];
  const float mean = tot / float(dim);
  float ss = 0.f;
  for (int d = threadIdx.x; d < dim; d += blockDim.x) { const float c = pooled[d] - mean; ss += c * c; }
  ss = warp_sum(ss);
  if (lane == 0) red[8 + warp] = ss;
  __syncthreads();
  float tot2 = 0.f;
  for (int w = 0; w < 8; ++w) tot2 += red[8 + w];
  const float rstd = rsqrtf(tot2 / float(dim) + eps);
  for (int d = threadIdx.x; d < dim; d += blockDim.x) {
    const float o = (pooled[d] - mean) * rstd * scale[d] + bias[d];
    if constexpr (kDT != DT_F32) reinterpret_cast<uint16_t*>(y)[int64_t(b) * dim + d] = cvt16<kDT>(o);
    else reinterpret_cast<float*>(y)[int64_t(b) * dim + d] = o;
  }
}

// ----------------------------------------------------------- weight pack (K7)
// W fp32 [K, N] (flax kernel) -> Wt bf16 [N, Kpad], zero padded along K.
template <int kDT>
__global__ void __launch_bounds__(256)
pack_weight_kernel(const float* __restrict__ W, uint16_t* __restrict__ Wt, int K, int N, int Kpad) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, n = n0 + tx;
    tile[r][tx] = (k < K && n < N) ? W[int64_t(k) * N + n] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int n = n0 + r, k = k0 + tx;
    if (n < N && k < Kpad) Wt[int64_t(n) * Kpad + k] = cvt16<kDT>(tile[tx][r]);
  }
}

// ------------------------------------------------ LayerNorm fold, weight side
// (gemm_tc.cu header)  Ws[k, n] = gamma[k] W[k, n]; d[n] = sum_k beta[k] W[k, n] (+ bias[n]); c[n] = sum_k of the
// 16-bit ROUNDED packed row Wt[n, :].  Run per weight load and after every optimiser step (the in-place refresh).
// One CTA per 32 columns: all eight warps stream FOLD_ROWS-row slabs of W (coalesced over n) into shared memory and
// write Ws, then warp 0 carries each column's d chain through the slab -- the same fmaf sequence k = 0 .. K-1 as one
// thread per column, with the loads of a whole CTA in flight instead of one per thread.
constexpr int FOLD_ROWS = 128;
__global__ void __launch_bounds__(256)
fold_scale_kernel(const float* __restrict__ W, const float* __restrict__ gamma, const float* __restrict__ beta,
                  const float* __restrict__ bias, float* __restrict__ Ws, float* __restrict__ d, int K, int N) {
  __shared__ float tile[FOLD_ROWS][33];
  __shared__ float bs[FOLD_ROWS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + lane;
  float acc = (n < N && bias) ? bias[n] : 0.f;
  for (int k0 = 0; k0 < K; k0 += FOLD_ROWS) {
    const int rows = min(FOLD_ROWS, K - k0);
    for (int r = warp; r < rows; r += 8) {
      const int64_t i = int64_t(k0 + r) * N + n;
      const float w = n < N ? W[i] : 0.f;
      if (n < N) Ws[i] = gamma[k0 + r] * w;
      tile[r][lane] = w;
    }
    for (int r = threadIdx.x; r < rows; r += blockDim.x) bs[r] = beta[k0 + r];
    __syncthreads();
    if (warp == 0)
      for (int r = 0; r < rows; ++r) acc = fmaf(bs[r], tile[r][lane], acc);
    __syncthreads();
  }
  if (warp == 0 && n < N) d[n] = acc;
}
// ------------------------------------------------ E4M3 weight quantisation (fp8)
// W fp32 [K, N] -> Wt E4M3 [N, Kpad], scale[n] = amax_k |W[k, n]| / 448 (1 for an all-zero column).  One CTA per 32
// columns like fold_scale_kernel: the eight warps stream rows (coalesced over n) for the column maxima, then 32 x 32
// tiles are transposed through shared memory so that the byte rows of Wt are written along k.
__global__ void __launch_bounds__(256)
quantize_e4m3_kernel(const float* __restrict__ W, uint8_t* __restrict__ Wt, float* __restrict__ scale, int K, int N, int Kpad) {
  __shared__ float tile[32][33];
  __shared__ float red[8][32];
  __shared__ float sc[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n0 = blockIdx.x * 32, n = n0 + lane;
  float amax = 0.f;
  if (n < N)
    for (int k = warp; k < K; k += 8) amax = fmaxf(amax, fabsf(W[int64_t(k) * N + n]));
  red[warp][lane] = amax;
  __syncthreads();
  if (warp == 0) {
    for (int w = 1; w < 8; ++w) amax = fmaxf(amax, red[w][lane]);
    const float s = amax > 0.f ? amax / 448.0f : 1.0f;
    sc[lane] = s;
    if (n < N) scale[n] = s;
  }
  __syncthreads();
  for (int k0 = 0; k0 < Kpad; k0 += 32) {
    for (int r = warp; r < 32; r += 8) {
      const int k = k0 + r;
      tile[r][lane] = (k < K && n < N) ? __fdiv_rn(W[int64_t(k) * N + n], sc[lane]) : 0.f;
    }
    __syncthreads();
    for (int r = warp; r < 32; r += 8) {   // row n0 + r of Wt, bytes k0 + lane
      const int nn = n0 + r, k = k0 + lane;
      if (nn < N && k < Kpad) Wt[int64_t(nn) * Kpad + k] = uint8_t(pack4_e4m3(tile[lane][r], 0.f, 0.f, 0.f) & 0xFFu);
    }
    __syncthreads();
  }
}

template <int kDT>
__global__ void __launch_bounds__(256)
fold_rowsum16_kernel(const uint16_t* __restrict__ Wt, float* __restrict__ c, int N, int Kpad) {
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;   // one warp per packed row
  if (n >= N) return;
  float acc = 0.f;
  for (int k = lane; k < Kpad; k += 32) acc += to_f32<kDT>(Wt[int64_t(n) * Kpad + k]);
  acc = warp_sum(acc);
  if (lane == 0) c[n] = acc;
}

// ------------------------------------------------------ fp32 SIMT GEMM (mode)
__device__ __forceinline__ float gelu_tanh_exact(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  return 0.5f * x * (1.0f + tanhf(k0 * (x + k1 * x * x * x)));
}

template <int kEpi>
__global__ void __launch_bounds__(256)
gemm_f32_kernel(const float* __restrict__ A, const float* __restrict__ W,
                const float* __restrict__ bias, float* __restrict__ C, int M, int N, int K,
                const float* __restrict__ aux, int tpi, Dropout drop, int cls_off) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int a_row = tid >> 2, a_k = (tid & 3) * 4;     // 64 rows x 16 k
  const int b_k = tid >> 4, b_n = (tid & 15) * 4;      // 16 k x 64 n
  for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int m = m0 + a_row, k = k0 + a_k + e;
      As[a_k + e][a_row] = (m < M && k < K) ? A[int64_t(m) * K + k] : 0.f;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = k0 + b_k, n = n0 + b_n + e;
      Bs[b_k][b_n + e] = (k < K && n < N) ? W[int64_t(k) * N + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
    int64_t out_row = m;
    const float* pos_row = nullptr;
    if constexpr (kEpi == VITB200_EPI_PATCH_F32) {
      const int b = m / tpi, t = m - b * tpi;
      out_row = int64_t(b) * (tpi + cls_off) + cls_off + t;
      pos_row = aux + int64_t(cls_off + t) * N;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      if constexpr (kEpi != VITB200_EPI_STORE_16) v += bias[n];
      if constexpr (kEpi == VITB200_EPI_BIAS_GELU_16) v = gelu_tanh_exact(v);
      if constexpr (kEpi == VITB200_EPI_PATCH_F32) v += pos_row[n];
      if constexpr (kEpi == VITB200_EPI_BIAS_GELU_16 || kEpi == VITB200_EPI_BIAS_RESID_F32 ||
                    kEpi == VITB200_EPI_PATCH_F32) {
        if (drop.threshold != 0) {   // same sites and flat indices as the tensor-core epilogues
          const int64_t e = out_row * N + n;
          const uint4 r = philox4x32_10(static_cast<unsigned long long>(e) >> 2, drop.site, drop.key_lo, drop.key_hi);
          const uint32_t w = (e & 3) == 0 ? r.x : (e & 3) == 1 ? r.y : (e & 3) == 2 ? r.z : r.w;
          v = w < drop.threshold ? 0.f : v * drop.inv_keep;
        }
      }
      if constexpr (kEpi == VITB200_EPI_BIAS_RESID_F32) v += C[out_row * N + n];
      C[out_row * N + n] = v;
    }
  }
}

template <int kEpi>
int launch_gemm_f32_t(cudaStream_t st, const float* A, const float* W, const float* bias, float* C,
                      int M, int N, int K, const float* aux, int tpi, const Dropout& drop, int cls_off) {
  dim3 grid(ceil_div(N, 64), ceil_div(M, 64));
  gemm_f32_kernel<kEpi><<<grid, 256, 0, st>>>(A, W, bias, C, M, N, K, aux, tpi, drop, cls_off);
  VB_LAUNCH_CHECK("gemm_f32_kernel");
  return 0;
}

// -------------------------------------------------- fp32 attention (mode)
// One warp per query row; scores for the row live in shared memory.
__global__ void __launch_bounds__(256)
attention_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out, int T, int heads) {
  extern __shared__ float sh[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Tpad = (T + 31) & ~31;
  float* sc = sh + warp * (Tpad + 64);
  float* qs = sc + Tpad;
  const int bh = blockIdx.x, b = bh / heads, h = bh - b * heads;
  const int qi = blockIdx.y * 8 + warp;
  if (qi >= T) return;
  const int inner = heads * 64, ld = 3 * inner;
  const float* base = qkv + int64_t(b) * T * ld;
  const float* qrow = base + int64_t(qi) * ld + h * 64;
  qs[lane] = qrow[lane];
  qs[lane + 32] = qrow[lane + 32];
  __syncwarp();
  float mx = -INFINITY;
  for (int j = lane; j < T; j += 32) {
    const float4* kr = reinterpret_cast<const float4*>(base + int64_t(j) * ld + inner + h * 64);
    float d = 0.f;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const float4 kv = __ldg(kr + c);
      d = fmaf(qs[c * 4 + 0], kv.x, d); d = fmaf(qs[c * 4 + 1], kv.y, d);
      d = fmaf(qs[c * 4 + 2], kv.z, d); d = fmaf(qs[c * 4 + 3], kv.w, d);
    }
    d *= 0.125f;                       // dim_head ** -0.5, dim_head = 64 (vit.py:66)
    sc[j] = d;
    mx = fmaxf(mx, d);
  }
  mx = warp_max(mx);
  float sum = 0.f;
  for (int j = lane; j < T; j += 32) {
    const float e = expf(sc[j] - mx);
    sc[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  __syncwarp();
  float o0 = 0.f, o1 = 0.f;
  const float* vbase = base + 2 * inner + h * 64;
  for (int j = 0; j < T; ++j) {
    const float p = sc[j];
    o0 = fmaf(p, __ldg(vbase + int64_t(j) * ld + lane), o0);
    o1 = fmaf(p, __ldg(vbase + int64_t(j) * ld + lane + 32), o1);
  }
  const float inv = 1.f / sum;
  float* orow = out + (int64_t(b) * T + qi) * inner + h * 64;
  orow[lane] = o0 * inv;
  orow[lane + 32] = o1 * inv;
}

}  // namespace

// ------------------------------------------------------------------ launchers
#define VB_DT_DISPATCH(dt, CALL)                                                        \
  switch (dt) {                                                                        \
    case DT_F32: { constexpr int kDT = DT_F32; CALL; break; }                          \
    case DT_BF16: { constexpr int kDT = DT_BF16; CALL; break; }                        \
    case DT_F16: { constexpr int kDT = DT_F16; CALL; break; }                          \
    default: return fail(VITB200_ERR_INVALID, "dtype must be VITB200_DT_F32/BF16/F16"); \
  }

int launch_layernorm(cudaStream_t st, const float* x, const float* g, const float* b, void* y,
                     int rows, int dim, int out_dtype, float eps, float* copy, int64_t ldx) {
  if (rows <= 0 || dim <= 0) return fail(VITB200_ERR_INVALID, "layernorm: empty problem");
  if (ldx == 0) ldx = dim;
  if (ldx < dim || (copy != nullptr && ldx != dim)) return fail(VITB200_ERR_INVALID, "layernorm: bad row pitch of x");
  if (out_dtype == DT_E4M3) return launch_ln_t<DT_E4M3>(st, x, g, b, y, rows, dim, eps, copy, ldx);   // only this launcher takes E4M3
  VB_DT_DISPATCH(out_dtype, return launch_ln_t<kDT>(st, x, g, b, y, rows, dim, eps, copy, ldx));
  return 0;
}

int launch_patchify(cudaStream_t st, const float* images, void* patches, int batch, int H, int W,
                    int C, int ph, int pw, int Kpad, int out_dtype, int nchw, int tok_off) {
  if (batch <= 0 || H <= 0 || W <= 0 || C <= 0 || ph <= 0 || pw <= 0)
    return fail(VITB200_ERR_INVALID, "patchify: empty problem");
  if (H % ph != 0 || W % pw != 0)
    return fail(VITB200_ERR_INVALID, "patchify: image not divisible by patch (vit.py:133-134)");
  if (Kpad < ph * pw * C || (Kpad & 1))
    return fail(VITB200_ERR_INVALID, "patchify: Kpad must be even and >= ph*pw*C");
  if (!nchw && ((pw * C) & 3) == 0 && (Kpad & 3) == 0 && (reinterpret_cast<uintptr_t>(images) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(patches) & 15) == 0 && int64_t(batch) * H < (int64_t(1) << 31)) {
    const int n4 = (W * C) >> 2;
    const int threads = n4 >= 256 ? 256 : ((n4 + 31) / 32) * 32;
    VB_DT_DISPATCH(out_dtype, (launch_kernel(patchify_row4_kernel<kDT>, dim3(unsigned(std::min<int64_t>(int64_t(batch) * H, int64_t(sm_count()) * 8))), dim3(threads), 0, st, 1, images, patches, batch * H, H, W, C, ph, pw, Kpad, tok_off)));
    VB_LAUNCH_CHECK("patchify_row4_kernel");
    return 0;
  }
  if (!nchw && ((pw * C) & 1) == 0 && (reinterpret_cast<uintptr_t>(images) & 7) == 0) {
    const int64_t total = int64_t(batch) * H * ((W * C) >> 1);
    const int grid = int(std::min<int64_t>((total + 255) / 256, int64_t(sm_count()) * 16));
    VB_DT_DISPATCH(out_dtype, (launch_kernel(patchify_rows_kernel<kDT>, dim3(grid), dim3(256), 0, st, 1, images, patches, batch, H, W, C, ph, pw, Kpad, tok_off)));
    VB_LAUNCH_CHECK("patchify_rows_kernel");
    return 0;
  }
  const int64_t total = int64_t(batch) * (H / ph) * (W / pw) * (Kpad / 2);
  const int grid = int(std::min<int64_t>((total + 255) / 256, int64_t(sm_count()) * 16));
  VB_DT_DISPATCH(out_dtype, (launch_kernel(patchify_kernel<kDT>, dim3(grid), dim3(256), 0, st, 1, images, patches, batch, H, W, C, ph, pw, Kpad, nchw, tok_off)));
  VB_LAUNCH_CHECK("patchify_kernel");
  return 0;
}

int launch_unpatchify(cudaStream_t st, const float* patches, float* images, int batch, int H, int W, int C, int ph,
                      int pw, int Kpad, int nchw, int tok_off) {
  if (batch <= 0 || H <= 0 || W <= 0 || C <= 0 || ph <= 0 || pw <= 0)
    return fail(VITB200_ERR_INVALID, "unpatchify: empty problem");
  if (H % ph != 0 || W % pw != 0)
    return fail(VITB200_ERR_INVALID, "unpatchify: image not divisible by patch (vit.py:133-134)");
  if (Kpad < ph * pw * C) return fail(VITB200_ERR_INVALID, "unpatchify: Kpad must be >= ph*pw*C");
  if (!nchw && ((pw * C) & 3) == 0 && (Kpad & 3) == 0 && (reinterpret_cast<uintptr_t>(images) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(patches) & 15) == 0 && int64_t(batch) * H < (int64_t(1) << 31)) {
    const int n4 = (W * C) >> 2;
    const int threads = n4 >= 256 ? 256 : ((n4 + 31) / 32) * 32;
    VB_CUDA(launch_kernel(unpatchify_row4_kernel, dim3(unsigned(std::min<int64_t>(int64_t(batch) * H, int64_t(sm_count()) * 8))),
                          dim3(threads), 0, st, 1, patches, images, batch * H, H, W, C, ph, pw, Kpad, tok_off));
    VB_LAUNCH_CHECK("unpatchify_row4_kernel");
    return 0;
  }
  const int64_t total = int64_t(batch) * H * W * C;
  const int grid = int(std::min<int64_t>((total + 255) / 256, int64_t(sm_count()) * 16));
  VB_CUDA(launch_kernel(unpatchify_kernel, dim3(grid), dim3(256), 0, st, 1, patches, images, batch, H, W, C, ph, pw, Kpad,
                        nchw, tok_off));
  VB_LAUNCH_CHECK("unpatchify_kernel");
  return 0;
}

int launch_cls_rows(cudaStream_t st, const float* cls, const float* pos, float* x, int batch, int T,
                    int dim, const Dropout& drop) {
  const int64_t total = int64_t(batch) * dim;
  VB_CUDA(launch_kernel(cls_rows_kernel, dim3(unsigned((total + 255) / 256)), dim3(256), 0, st, 1, cls, pos, x, batch, T, dim, drop));
  VB_LAUNCH_CHECK("cls_rows_kernel");
  return 0;
}

int launch_pool_layernorm(cudaStream_t st, const float* x, const float* g, const float* b, void* y,
                          int batch, int T, int dim, int pool, int out_dtype, float eps) {
  if (pool != VITB200_POOL_CLS && pool != VITB200_POOL_MEAN)
    return fail(VITB200_ERR_INVALID, "pool must be cls or mean (vit.py:137)");
  const size_t smem = (size_t(dim) + 16) * sizeof(float);
  VB_DT_DISPATCH(out_dtype, (launch_kernel(pool_layernorm_kernel<kDT>, dim3(batch), dim3(256), smem, st, 1, x, g, b, y, T, dim, pool, eps)));
  VB_LAUNCH_CHECK("pool_layernorm_kernel");
  return 0;
}

int launch_pack_weight(cudaStream_t st, const float* W, void* Wt, int K, int N, int Kpad, int dtype) {
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(VITB200_ERR_INVALID, "pack_weight: dtype must be bf16 or fp16");
  dim3 grid(ceil_div(Kpad, 32), ceil_div(N, 32));
  if (dtype == DT_BF16) pack_weight_kernel<DT_BF16><<<grid, 256, 0, st>>>(W, static_cast<uint16_t*>(Wt), K, N, Kpad);
  else pack_weight_kernel<DT_F16><<<grid, 256, 0, st>>>(W, static_cast<uint16_t*>(Wt), K, N, Kpad);
  VB_LAUNCH_CHECK("pack_weight_kernel");
  return 0;
}

int launch_quantize_weight_e4m3(cudaStream_t st, const float* W, uint8_t* Wt, float* scale, int K, int N, int Kpad) {
  if (K <= 0 || N <= 0 || Kpad < K || (Kpad % 16) != 0)
    return fail(VITB200_ERR_INVALID, "quantize_weight_e4m3: K, N > 0 and Kpad >= K, a multiple of 16");
  quantize_e4m3_kernel<<<ceil_div(N, 32), 256, 0, st>>>(W, Wt, scale, K, N, Kpad);
  VB_LAUNCH_CHECK("quantize_e4m3_kernel");
  return 0;
}

int launch_fold_layernorm(cudaStream_t st, const float* W, const float* gamma, const float* beta, const float* bias,
                          void* Wt, float* c, float* d, int K, int N, int Kpad, int dtype, float* scratch) {
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(VITB200_ERR_INVALID, "fold_layernorm: dtype must be bf16 or fp16");
  if (K <= 0 || N <= 0 || Kpad < K) return fail(VITB200_ERR_INVALID, "fold_layernorm: bad shape");
  fold_scale_kernel<<<ceil_div(N, 32), 256, 0, st>>>(W, gamma, beta, bias, scratch, d, K, N);
  VB_LAUNCH_CHECK("fold_scale_kernel");
  int rc = launch_pack_weight(st, scratch, Wt, K, N, Kpad, dtype);
  if (rc) return rc;
  if (dtype == DT_BF16) fold_rowsum16_kernel<DT_BF16><<<ceil_div(N, 8), 256, 0, st>>>(static_cast<const uint16_t*>(Wt), c, N, Kpad);
  else fold_rowsum16_kernel<DT_F16><<<ceil_div(N, 8), 256, 0, st>>>(static_cast<const uint16_t*>(Wt), c, N, Kpad);
  VB_LAUNCH_CHECK("fold_rowsum16_kernel");
  return 0;
}

int launch_gemm_f32(cudaStream_t st, const float* A, const float* W, const float* bias, float* C,
                    int M, int N, int K, int epilogue, const float* aux, int tpi, const Dropout& drop,
                    int cls_off) {
  if (M <= 0 || N <= 0 || K <= 0) return fail(VITB200_ERR_INVALID, "gemm_f32: empty problem");
  if (epilogue != VITB200_EPI_STORE_16 && bias == nullptr)
    return fail(VITB200_ERR_INVALID, "gemm_f32: epilogue needs a bias");
  switch (epilogue) {
    case VITB200_EPI_STORE_16: return launch_gemm_f32_t<VITB200_EPI_STORE_16>(st, A, W, bias, C, M, N, K, aux, tpi, drop, cls_off);
    case VITB200_EPI_BIAS_GELU_16: return launch_gemm_f32_t<VITB200_EPI_BIAS_GELU_16>(st, A, W, bias, C, M, N, K, aux, tpi, drop, cls_off);
    case VITB200_EPI_BIAS_RESID_F32: return launch_gemm_f32_t<VITB200_EPI_BIAS_RESID_F32>(st, A, W, bias, C, M, N, K, aux, tpi, drop, cls_off);
    case VITB200_EPI_BIAS_F32: return launch_gemm_f32_t<VITB200_EPI_BIAS_F32>(st, A, W, bias, C, M, N, K, aux, tpi, drop, cls_off);
    case VITB200_EPI_PATCH_F32:
      if (aux == nullptr || tpi <= 0) return fail(VITB200_ERR_INVALID, "gemm_f32: PATCH epilogue needs pos_embedding and tokens");
      return launch_gemm_f32_t<VITB200_EPI_PATCH_F32>(st, A, W, bias, C, M, N, K, aux, tpi, drop, cls_off);
    default: return fail(VITB200_ERR_INVALID, "gemm_f32: unknown epilogue");
  }
}

int launch_attention_f32(cudaStream_t st, const float* qkv, float* out, int batch, int T, int heads) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention_f32: empty problem");
  const int Tpad = (T + 31) & ~31;
  const size_t smem = size_t(8) * (Tpad + 64) * sizeof(float);
  static PerDevice<bool> configured_on;   // the smem opt-in is per (function, device)
  if (bool& configured = configured_on.here(); !configured && smem > 48 * 1024) {
    VB_CUDA(cudaFuncSetAttribute(attention_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured = true;
  }
  if (smem > 200 * 1024) return fail(VITB200_ERR_UNSUPPORTED, "attention_f32: sequence too long");
  dim3 grid(batch * heads, ceil_div(T, 8));
  attention_f32_kernel<<<grid, 256, smem, st>>>(qkv, out, T, heads);
  VB_LAUNCH_CHECK("attention_f32_kernel");
  return 0;
}

}  // namespace vb
