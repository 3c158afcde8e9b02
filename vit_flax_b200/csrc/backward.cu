// backward.cu -- kernels of the backward pass (SURVEY.md section 8f-4): everything that is not a GEMM.
//
// The reference never differentiates its forward (nothing in vit_flax trains), so there is no
// reference code to cite beyond the forward lines each kernel is the adjoint of:
//   (the attention adjoint, vit.py:69-79, is attention_bwd_tc5.cu; launch_attention_bwd below only routes to it)
//   ln_bwd_kernel          adjoint of nn.LayerNorm() (vit.py:31,163)
//   gelu_fwd / gelu_bwd    nn.gelu (tanh form, vit.py:49) on the stored pre-activation
//   pool_ln_bwd_kernel     adjoint of vit.py:159-163 (cls / mean pool + LayerNorm)
//   token_grad kernels     adjoint of vit.py:151-153 (cls concat + pos_embedding broadcast over the batch)
//   transpose16 / cast16 / colsum: operand preparation for the weight-gradient GEMMs and the bias gradients
// The GEMMs (dgrad: dX = dY W^T, wgrad: dW = X^T dY) run on the tcgen05 kernel of gemm_tc.cu.
#include <algorithm>
#include <cstdlib>

#include "common.h"
#include "ptx.cuh"

namespace vb {

namespace {

template <int kDT>
__device__ __forceinline__ void unpack2(uint32_t v, float& lo, float& hi) {
  lo = to_f32<kDT>(uint16_t(v & 0xFFFFu));
  hi = to_f32<kDT>(uint16_t(v >> 16));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------ elementwise
template <int kDT>
__global__ void __launch_bounds__(256)
cast16_kernel(const float* __restrict__ x, uint16_t* __restrict__ y, int64_t n8) {   // n8 = elements / 8
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n8; i += int64_t(gridDim.x) * blockDim.x) {
    const float4 a = reinterpret_cast<const float4*>(x)[2 * i], b = reinterpret_cast<const float4*>(x)[2 * i + 1];
    uint4 o;
    o.x = pack2<kDT>(a.x, a.y); o.y = pack2<kDT>(a.z, a.w);
    o.z = pack2<kDT>(b.x, b.y); o.w = pack2<kDT>(b.z, b.w);
    reinterpret_cast<uint4*>(y)[i] = o;
  }
}

// tanh.approx (one MUFU op, 2^-11 relative) as in the forward GEMM epilogue: with tanhf these passes were
// issue-bound (72 % issue-slot utilisation, profiles/r01_backward.md) instead of HBM-bound
__device__ __forceinline__ float gelu_tanh_ref(float x) {   // nn.gelu default (vit.py:49)
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  return 0.5f * x * (1.0f + tanh_approx(k0 * x * fmaf(k1 * x, x, 1.0f)));
}
__device__ __forceinline__ float gelu_tanh_grad(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  const float t = tanh_approx(k0 * x * fmaf(k1 * x, x, 1.0f));
  return 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * k0 * fmaf(3.0f * k1 * x, x, 1.0f);
}

template <int kDT, bool kBwd>
__global__ void __launch_bounds__(256)
gelu_kernel(const uint16_t* __restrict__ pre, const uint16_t* __restrict__ dhid, uint16_t* __restrict__ out, int64_t n8,
            Dropout drop) {   // forward: nn.Dropout behind the GELU (vit.py:50), flat element index = 8 i
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n8; i += int64_t(gridDim.x) * blockDim.x) {
    const uint4 p = reinterpret_cast<const uint4*>(pre)[i];
    uint4 d = make_uint4(0, 0, 0, 0);
    if constexpr (kBwd) d = reinterpret_cast<const uint4*>(dhid)[i];
    const uint32_t pw[4] = {p.x, p.y, p.z, p.w}, dw[4] = {d.x, d.y, d.z, d.w};
    uint32_t ow[4];
    float v[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a, b;
      unpack2<kDT>(pw[j], a, b);
      if constexpr (kBwd) {
        float da, db;
        unpack2<kDT>(dw[j], da, db);
        v[2 * j] = da * gelu_tanh_grad(a);
        v[2 * j + 1] = db * gelu_tanh_grad(b);
      } else {
        v[2 * j] = gelu_tanh_ref(a);
        v[2 * j + 1] = gelu_tanh_ref(b);
      }
    }
    if (drop.threshold != 0) {
      dropout4(drop, i * 8, v[0], v[1], v[2], v[3]);
      dropout4(drop, i * 8 + 4, v[4], v[5], v[6], v[7]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) ow[j] = pack2<kDT>(v[2 * j], v[2 * j + 1]);
    reinterpret_cast<uint4*>(out)[i] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
  }
}

// Fused row passes with a column sum (the bias gradients ride along with a pass that is needed anyway):
//   MODE 0: y16 = cast(x32),                      sums += x32          (dy for the GEMMs + db of to_out / FF Dense_1)
//   MODE 1: out16 = dhid16 * gelu'(pre16),        sums += out16        (gelu backward + db of FF Dense_0)
// A thread owns 8 consecutive columns and walks rows blockIdx.y * 8 + ty, + 8 gridDim.y, ...; a block covers
// 256 columns; the 8 row lanes of a block meet in shared memory, then one atomic per column and block.
template <int kDT, int MODE>
__global__ void __launch_bounds__(256)
rowpass_colsum_kernel(const void* __restrict__ in0, const uint16_t* __restrict__ in1, uint16_t* __restrict__ out,
                      float* __restrict__ sums, int rows, int cols, Dropout drop) {   // drop: the mask of the forward's nn.Dropout
                                                                                      // at this tensor (flat index r * cols + c), replayed
  __shared__ float red[8][256];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 256 + tx * 8;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (c < cols) {
    for (int r = blockIdx.y * 8 + ty; r < rows; r += gridDim.y * 8) {
      const int64_t o = int64_t(r) * cols + c;
      float v[8];
      if constexpr (MODE == 0) {
        const float4 a = *reinterpret_cast<const float4*>(static_cast<const float*>(in0) + o);
        const float4 b = *reinterpret_cast<const float4*>(static_cast<const float*>(in0) + o + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
      } else {
        const uint4 p = *reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(in0) + o);
        const uint4 d = *reinterpret_cast<const uint4*>(in1 + o);
        const uint32_t pw[4] = {p.x, p.y, p.z, p.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float a, b, da, db;
          unpack2<kDT>(pw[j], a, b);
          unpack2<kDT>(dw[j], da, db);
          v[2 * j] = da * gelu_tanh_grad(a);
          v[2 * j + 1] = db * gelu_tanh_grad(b);
        }
      }
      if (drop.threshold != 0) {
        dropout4(drop, o, v[0], v[1], v[2], v[3]);
        dropout4(drop, o + 4, v[4], v[5], v[6], v[7]);
      }
      uint4 w;
      w.x = pack2<kDT>(v[0], v[1]); w.y = pack2<kDT>(v[2], v[3]); w.z = pack2<kDT>(v[4], v[5]); w.w = pack2<kDT>(v[6], v[7]);
      *reinterpret_cast<uint4*>(out + o) = w;
      if constexpr (MODE == 1) {   // the bias gradient is the sum of what the GEMMs will see: the rounded values
        unpack2<kDT>(w.x, v[0], v[1]); unpack2<kDT>(w.y, v[2], v[3]); unpack2<kDT>(w.z, v[4], v[5]); unpack2<kDT>(w.w, v[6], v[7]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += v[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[ty][tx * 8 + j] = acc[j];
  __syncthreads();
  const int col = blockIdx.x * 256 + threadIdx.x;
  if (col < cols) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += red[j][threadIdx.x];
    atomicAdd(sums + col, t);
  }
}

// x[i] = mask(i) ? x[i] / keep : 0 in place (the embedding dropout, vit.py:155, in the backward pass)
__global__ void __launch_bounds__(256)
mask_inplace_kernel(float* __restrict__ x, int64_t n4, Dropout drop) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n4; i += int64_t(gridDim.x) * blockDim.x) {
    float4 v = reinterpret_cast<float4*>(x)[i];
    dropout4(drop, i * 4, v.x, v.y, v.z, v.w);
    reinterpret_cast<float4*>(x)[i] = v;
  }
}

// out[c, r] = in[r, c] for r < rows, 0 for rows <= r < rows_pad  (16-bit elements, 64x64 tiles)
__global__ void __launch_bounds__(256)
transpose16_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, int rows, int cols, int rows_pad) {
  __shared__ uint16_t tile[64][66];
  const int r0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 32 x 8
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = r0 + ty + i * 8, c = c0 + 2 * tx;
    uint32_t v = 0;
    if (r < rows && c < cols) v = *reinterpret_cast<const uint32_t*>(in + int64_t(r) * cols + c);   // cols is even
    tile[ty + i * 8][2 * tx] = uint16_t(v & 0xFFFFu);
    tile[ty + i * 8][2 * tx + 1] = uint16_t(v >> 16);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = c0 + ty + i * 8, r = r0 + 2 * tx;
    if (c < cols && r < rows_pad) {
      const uint32_t v = uint32_t(tile[2 * tx][ty + i * 8]) | (uint32_t(tile[2 * tx + 1][ty + i * 8]) << 16);
      *reinterpret_cast<uint32_t*>(out + int64_t(c) * rows_pad + r) = v;      // rows_pad is even
    }
  }
}

// out[c] += sum_r in[r, c]   (bias gradients); two columns per thread, rows strided over blockIdx.y
template <int kDT>
__global__ void __launch_bounds__(256)
colsum_kernel(const void* __restrict__ in, float* __restrict__ out, int rows, int cols) {
  __shared__ float red[8][64];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + 2 * tx;
  float a = 0.f, b = 0.f;
  if (c < cols) {
    for (int r = blockIdx.y * 8 + ty; r < rows; r += gridDim.y * 8) {
      if constexpr (kDT == DT_F32) {
        const float2 v = *reinterpret_cast<const float2*>(static_cast<const float*>(in) + int64_t(r) * cols + c);
        a += v.x; b += v.y;
      } else {
        float x, y;
        unpack2<kDT>(*reinterpret_cast<const uint32_t*>(static_cast<const uint16_t*>(in) + int64_t(r) * cols + c), x, y);
        a += x; b += y;
      }
    }
  }
  red[ty][2 * tx] = a;
  red[ty][2 * tx + 1] = b;
  __syncthreads();
  if (ty == 0 && c < cols) {
#pragma unroll
    for (int j = 1; j < 8; ++j) { a += red[j][2 * tx]; b += red[j][2 * tx + 1]; }
    atomicAdd(out + c, a);
    atomicAdd(out + c + 1, b);
  }
}

// ------------------------------------------------------------------ LayerNorm backward
// dx[r,:] (+)= rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma;  dgamma += sum_r dy * xhat,
// dbeta += sum_r dy.  One warp per row, float4 / 8-byte accesses: lane owns columns 4 (lane + 32 k) .. +3,
// k < KV (dim <= 128 KV).  The kernel is a pure HBM stream (14 bytes per element), so what matters is
// bytes in flight: the loads of the warp's NEXT row (x, dy, dx) are issued before the current row is
// reduced, and dgamma / dbeta accumulate in a warp-private shared-memory strip (no atomics, no
// registers) that the block folds into one atomic per column at the end.
template <int kDT, int KV>
__global__ void __launch_bounds__(128)
ln_bwd_kernel(const uint16_t* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
              float* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta, int rows, int dim,
              float eps, int accumulate, uint16_t* __restrict__ dx16, float* __restrict__ dbias_next, Dropout drop) {
  // dx16 != null: the new dx is also what the NEXT stage's GEMMs consume, so it leaves here as 16 bits too
  // (with that stage's nn.Dropout mask replayed) and its column sums are that stage's bias gradient --
  // this replaces a separate cast + column-sum pass over dx
  extern __shared__ float4 acc_sm[];        // [warps][3][dim / 4]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int nvec = dim >> 2;
  float4* ag = acc_sm + size_t(warp) * 3 * nvec;
  float4* ab = ag + nvec;
  float4* an = ab + nvec;
  for (int i = lane; i < 3 * nvec; i += 32) ag[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
  const float inv_d = 1.0f / float(dim);
  const int stride = gridDim.x * nw;
  int r = blockIdx.x * nw + warp;
  float4 nx[KV], no[KV];
  uint2 nd[KV];
  auto fetch = [&](int row) {
#pragma unroll
    for (int k = 0; k < KV; ++k) {
      const int c = lane + 32 * k;
      if (c < nvec && row < rows) {
        nx[k] = reinterpret_cast<const float4*>(x + int64_t(row) * dim)[c];
        nd[k] = reinterpret_cast<const uint2*>(dy + int64_t(row) * dim)[c];
        no[k] = accumulate ? reinterpret_cast<const float4*>(dx + int64_t(row) * dim)[c] : make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        nx[k] = no[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        nd[k] = make_uint2(0u, 0u);
      }
    }
  };
  fetch(r);
  for (; r < rows; r += stride) {
    float4 xv[KV], dv[KV], ov[KV];
#pragma unroll
    for (int k = 0; k < KV; ++k) {
      xv[k] = nx[k];
      ov[k] = no[k];
      unpack2<kDT>(nd[k].x, dv[k].x, dv[k].y);
      unpack2<kDT>(nd[k].y, dv[k].z, dv[k].w);
    }
    fetch(r + stride);                        // in flight while this row is reduced
    float s = 0.f, ss = 0.f;
#pragma unroll
    for (int k = 0; k < KV; ++k) {
      s += (xv[k].x + xv[k].y) + (xv[k].z + xv[k].w);
      ss += (xv[k].x * xv[k].x + xv[k].y * xv[k].y) + (xv[k].z * xv[k].z + xv[k].w * xv[k].w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {       // the two reductions share their shuffle latency
      s += __shfl_xor_sync(0xffffffffu, s, o);
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    const float mean = s * inv_d;
    const float rstd = rsqrtf(fmaxf(0.f, ss * inv_d - mean * mean) + eps);   // flax: var = max(0, E[x^2] - E[x]^2)
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int k = 0; k < KV; ++k) {
      const int c = lane + 32 * k;
      if (c < nvec) {
        const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + c);
        xv[k].x = (xv[k].x - mean) * rstd; xv[k].y = (xv[k].y - mean) * rstd;
        xv[k].z = (xv[k].z - mean) * rstd; xv[k].w = (xv[k].w - mean) * rstd;
        float4 g4 = ag[c], b4 = ab[c];
        g4.x += dv[k].x * xv[k].x; g4.y += dv[k].y * xv[k].y; g4.z += dv[k].z * xv[k].z; g4.w += dv[k].w * xv[k].w;
        b4.x += dv[k].x; b4.y += dv[k].y; b4.z += dv[k].z; b4.w += dv[k].w;
        ag[c] = g4;
        ab[c] = b4;
        dv[k].x *= gm.x; dv[k].y *= gm.y; dv[k].z *= gm.z; dv[k].w *= gm.w;      // g = dy * gamma
        a += (dv[k].x + dv[k].y) + (dv[k].z + dv[k].w);
        b += (dv[k].x * xv[k].x + dv[k].y * xv[k].y) + (dv[k].z * xv[k].z + dv[k].w * xv[k].w);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    a *= inv_d;
    b *= inv_d;
    float4* dxr = reinterpret_cast<float4*>(dx + int64_t(r) * dim);
#pragma unroll
    for (int k = 0; k < KV; ++k) {
      const int c = lane + 32 * k;
      if (c < nvec) {
        float4 v;
        v.x = ov[k].x + rstd * (dv[k].x - a - xv[k].x * b); v.y = ov[k].y + rstd * (dv[k].y - a - xv[k].y * b);
        v.z = ov[k].z + rstd * (dv[k].z - a - xv[k].z * b); v.w = ov[k].w + rstd * (dv[k].w - a - xv[k].w * b);
        dxr[c] = v;
        if (dx16 != nullptr) {
          if (drop.threshold != 0) dropout4(drop, int64_t(r) * dim + 4 * c, v.x, v.y, v.z, v.w);
          uint2 w;
          w.x = pack2<kDT>(v.x, v.y);
          w.y = pack2<kDT>(v.z, v.w);
          reinterpret_cast<uint2*>(dx16 + int64_t(r) * dim)[c] = w;
          float4 s4 = an[c];
          s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
          an[c] = s4;
        }
      }
    }
  }
  __syncthreads();
  const float* accf = reinterpret_cast<const float*>(acc_sm);
  for (int i = threadIdx.x; i < dim; i += blockDim.x) {
    float tg = 0.f, tb = 0.f, tn = 0.f;
    for (int w = 0; w < nw; ++w) {
      tg += accf[size_t(w) * 3 * dim + i];
      tb += accf[size_t(w) * 3 * dim + dim + i];
      tn += accf[size_t(w) * 3 * dim + 2 * dim + i];
    }
    atomicAdd(dgamma + i, tg);
    atomicAdd(dbeta + i, tb);
    if (dbias_next != nullptr) atomicAdd(dbias_next + i, tn);
  }
}

// ------------------------------------------------------------------ head: pool + LayerNorm backward
// One block per image.  pooled = x[b, 0] (cls) or mean_t x[b, t]; dpl = gradient wrt LayerNorm(pooled).
// The gradient wrt the pooled vector replaces dpl (same buffer is fine: each block owns its row).
__global__ void __launch_bounds__(256)
pool_ln_bwd_kernel(const float* __restrict__ x, const float* dpl, const float* __restrict__ gamma,
                   float* dpl_out, float* __restrict__ dgamma, float* __restrict__ dbeta, int T, int dim,
                   int pool_mean, float eps) {
  extern __shared__ float sh[];          // pooled[dim], g[dim], red[64]
  float* pooled = sh;
  float* gv = sh + dim;
  float* red = sh + 2 * dim;
  const int b = blockIdx.x;
  const float* xb = x + int64_t(b) * T * dim;
  for (int c = threadIdx.x; c < dim; c += blockDim.x) {
    float v;
    if (pool_mean) {
      v = 0.f;
      for (int t = 0; t < T; ++t) v += xb[int64_t(t) * dim + c];
      v /= float(T);
    } else {
      v = xb[c];
    }
    pooled[c] = v;
  }
  __syncthreads();
  auto block_sum2 = [&](float& a, float& c2) {
    a = warp_sum(a);
    c2 = warp_sum(c2);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) { red[w] = a; red[32 + w] = c2; }
    __syncthreads();
    float ra = 0.f, rc = 0.f;
    for (int i = 0; i < int(blockDim.x >> 5); ++i) { ra += red[i]; rc += red[32 + i]; }
    a = ra;
    c2 = rc;
  };
  float s = 0.f, ss = 0.f;
  for (int c = threadIdx.x; c < dim; c += blockDim.x) { s += pooled[c]; ss += pooled[c] * pooled[c]; }
  block_sum2(s, ss);
  const float mean = s / float(dim);
  const float rstd = rsqrtf(fmaxf(0.f, ss / float(dim) - mean * mean) + eps);
  float a = 0.f, bb = 0.f;
  for (int c = threadIdx.x; c < dim; c += blockDim.x) {
    const float xh = (pooled[c] - mean) * rstd, d = dpl[int64_t(b) * dim + c], g = d * gamma[c];
    pooled[c] = xh;
    gv[c] = g;
    a += g;
    bb += g * xh;
    atomicAdd(dgamma + c, d * xh);
    atomicAdd(dbeta + c, d);
  }
  block_sum2(a, bb);
  a /= float(dim);
  bb /= float(dim);
  __syncthreads();
  for (int c = threadIdx.x; c < dim; c += blockDim.x) gv[c] = rstd * (gv[c] - a - pooled[c] * bb) * (pool_mean ? 1.0f / float(T) : 1.0f);
  __syncthreads();
  // the pooled gradient goes back over dpl; pool_scatter_kernel spreads it over the image's token rows
  for (int c = threadIdx.x; c < dim; c += blockDim.x) dpl_out[int64_t(b) * dim + c] = gv[c];
}

// dx[b, t, :] = pooled gradient of image b for every t (mean pool, already divided by T) or for t = 0 only (cls), else 0
__global__ void __launch_bounds__(256)
pool_scatter_kernel(const float* __restrict__ dpooled, float* __restrict__ dx, int64_t total4, int T, int dim, int pool_mean) {
  const int per_row = dim >> 2;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total4; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t row = i / per_row;
    const int c4 = int(i - row * per_row);
    const int64_t b = row / T;
    const int t = int(row - b * T);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (pool_mean || t == 0) v = reinterpret_cast<const float4*>(dpooled + b * dim)[c4];
    reinterpret_cast<float4*>(dx)[i] = v;
  }
}

// head Dense backward (fp32, tiny): dW[d, c] += sum_b pl[b, d] dl[b, c];  dpl[b, d] = sum_c dl[b, c] W[d, c]
__global__ void __launch_bounds__(256)
head_wgrad_kernel(const float* __restrict__ pl, const float* __restrict__ dl, float* __restrict__ dW, int batch,
                  int dim, int classes) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, d = blockIdx.y;
  if (c >= classes) return;
  float acc = 0.f;
  for (int b = 0; b < batch; ++b) acc += pl[int64_t(b) * dim + d] * dl[int64_t(b) * classes + c];
  dW[int64_t(d) * classes + c] += acc;
}
__global__ void __launch_bounds__(256)
head_dgrad_kernel(const float* __restrict__ dl, const float* __restrict__ W, float* __restrict__ dpl, int batch,
                  int dim, int classes) {
  // one warp per (b, d): lanes stride over the classes
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= batch * dim) return;
  const int b = gw / dim, d = gw - b * dim;
  float acc = 0.f;
  for (int c = lane; c < classes; c += 32) acc += dl[int64_t(b) * classes + c] * W[int64_t(d) * classes + c];
  acc = warp_sum(acc);
  if (lane == 0) dpl[gw] = acc;
}

// ------------------------------------------------------------------ token gradients
// dpos[t, d] += sum_b dx[b, t, d]
__global__ void __launch_bounds__(256)
pos_grad_kernel(const float* __restrict__ dx, float* __restrict__ dpos, int batch, int T, int dim) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (d >= dim) return;
  float acc = 0.f;
  for (int b = 0; b < batch; ++b) acc += dx[(int64_t(b) * T + t) * dim + d];
  dpos[int64_t(t) * dim + d] += acc;
}
// after pos_grad on a zeroed dpos: dcls = dpos[0] (cls_off = 1), dbias = sum_{t >= cls_off} dpos[t]; the token rows
// are split over blockIdx.y (one atomic per column and slice)
__global__ void __launch_bounds__(256)
cls_bias_grad_kernel(const float* __restrict__ dpos, float* __restrict__ dcls, float* __restrict__ dbias, int T,
                     int dim, int cls_off) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= dim) return;
  float acc = 0.f;
  for (int t = cls_off + blockIdx.y; t < T; t += gridDim.y) acc += dpos[int64_t(t) * dim + d];
  atomicAdd(dbias + d, acc);
  if (blockIdx.y == 0 && cls_off && dcls) dcls[d] += dpos[d];
}

inline unsigned grid_for(int64_t work_items, int per_block) {
  return unsigned(std::min<int64_t>((work_items + per_block - 1) / per_block, int64_t(sm_count()) * 16));
}

}  // namespace

#define VB_DT_DISPATCH_ANY(dt, CALL)                                                    \
  switch (dt) {                                                                        \
    case DT_F32: { constexpr int kDT = DT_F32; CALL; break; }                          \
    case DT_BF16: { constexpr int kDT = DT_BF16; CALL; break; }                        \
    case DT_F16: { constexpr int kDT = DT_F16; CALL; break; }                          \
    default: return fail(VITB200_ERR_INVALID, "dtype must be VITB200_DT_F32/BF16/F16"); \
  }

#define VB_DT16_DISPATCH(dt, CALL)                                                     \
  switch (dt) {                                                                        \
    case DT_BF16: { constexpr int kDT = DT_BF16; CALL; break; }                        \
    case DT_F16: { constexpr int kDT = DT_F16; CALL; break; }                          \
    default: return fail(VITB200_ERR_INVALID, "dtype must be VITB200_DT_BF16/F16");   \
  }

int launch_cast16(cudaStream_t st, const float* x, void* y, int64_t n, int dtype) {
  if (n <= 0 || (n & 7)) return fail(VITB200_ERR_INVALID, "cast16: element count must be a positive multiple of 8");
  VB_DT16_DISPATCH(dtype, (cast16_kernel<kDT><<<grid_for(n / 8, 256), 256, 0, st>>>(x, static_cast<uint16_t*>(y), n / 8)));
  VB_LAUNCH_CHECK("cast16_kernel");
  return 0;
}

int launch_mask_inplace(cudaStream_t st, float* x, int64_t n, const Dropout& drop) {
  if (drop.threshold == 0) return 0;
  if (n <= 0 || (n & 3)) return fail(VITB200_ERR_INVALID, "mask_inplace: element count must be a positive multiple of 4");
  mask_inplace_kernel<<<grid_for(n / 4, 256), 256, 0, st>>>(x, n / 4, drop);
  VB_LAUNCH_CHECK("mask_inplace_kernel");
  return 0;
}

int launch_gelu_fwd(cudaStream_t st, const void* pre, void* hid, int64_t n, int dtype, const Dropout& drop) {
  if (n <= 0 || (n & 7)) return fail(VITB200_ERR_INVALID, "gelu: element count must be a positive multiple of 8");
  VB_DT16_DISPATCH(dtype, (gelu_kernel<kDT, false><<<grid_for(n / 8, 256), 256, 0, st>>>(
                              static_cast<const uint16_t*>(pre), nullptr, static_cast<uint16_t*>(hid), n / 8, drop)));
  VB_LAUNCH_CHECK("gelu_kernel(fwd)");
  return 0;
}

int launch_gelu_bwd(cudaStream_t st, const void* pre, const void* dhid, void* dpre, int64_t n, int dtype) {
  if (n <= 0 || (n & 7)) return fail(VITB200_ERR_INVALID, "gelu: element count must be a positive multiple of 8");
  VB_DT16_DISPATCH(dtype, (gelu_kernel<kDT, true><<<grid_for(n / 8, 256), 256, 0, st>>>(
                              static_cast<const uint16_t*>(pre), static_cast<const uint16_t*>(dhid),
                              static_cast<uint16_t*>(dpre), n / 8, Dropout())));
  VB_LAUNCH_CHECK("gelu_kernel(bwd)");
  return 0;
}

static dim3 rowpass_grid(int rows, int cols) {
  const int gx = (cols + 255) / 256;
  const int gy = std::max(1, std::min((rows + 7) / 8, std::max(1, 4 * sm_count() / gx)));
  return dim3(unsigned(gx), unsigned(gy));
}

int launch_cast16_colsum(cudaStream_t st, const float* x, void* y, float* sums, int rows, int cols, int dtype,
                         const Dropout& drop) {
  if (rows <= 0 || cols <= 0 || (cols & 7)) return fail(VITB200_ERR_INVALID, "cast16_colsum: cols must be a positive multiple of 8");
  VB_DT16_DISPATCH(dtype, (rowpass_colsum_kernel<kDT, 0><<<rowpass_grid(rows, cols), 256, 0, st>>>(
                              x, nullptr, static_cast<uint16_t*>(y), sums, rows, cols, drop)));
  VB_LAUNCH_CHECK("rowpass_colsum_kernel(cast)");
  return 0;
}

int launch_gelu_bwd_colsum(cudaStream_t st, const void* pre, const void* dhid, void* dpre, float* sums, int rows, int cols,
                           int dtype, const Dropout& drop) {
  if (rows <= 0 || cols <= 0 || (cols & 7)) return fail(VITB200_ERR_INVALID, "gelu_bwd_colsum: cols must be a positive multiple of 8");
  VB_DT16_DISPATCH(dtype, (rowpass_colsum_kernel<kDT, 1><<<rowpass_grid(rows, cols), 256, 0, st>>>(
                              pre, static_cast<const uint16_t*>(dhid), static_cast<uint16_t*>(dpre), sums, rows, cols, drop)));
  VB_LAUNCH_CHECK("rowpass_colsum_kernel(gelu_bwd)");
  return 0;
}

int launch_transpose16(cudaStream_t st, const void* in, void* out, int rows, int cols, int rows_pad) {
  if (rows <= 0 || cols <= 0 || rows_pad < rows || (cols & 1) || (rows_pad & 1))
    return fail(VITB200_ERR_INVALID, "transpose16: cols and rows_pad must be even, rows_pad >= rows");
  dim3 grid(unsigned((rows_pad + 63) / 64), unsigned((cols + 63) / 64));
  transpose16_kernel<<<grid, 256, 0, st>>>(static_cast<const uint16_t*>(in), static_cast<uint16_t*>(out), rows, cols, rows_pad);
  VB_LAUNCH_CHECK("transpose16_kernel");
  return 0;
}

int launch_colsum(cudaStream_t st, const void* in, float* out, int rows, int cols, int dtype) {
  if (rows <= 0 || cols <= 0 || (cols & 1)) return fail(VITB200_ERR_INVALID, "colsum: cols must be even");
  const int gx = (cols + 63) / 64;
  const int gy = std::max(1, std::min((rows + 63) / 64, std::max(1, 8 * sm_count() / gx)));
  dim3 grid{unsigned(gx), unsigned(gy)};
  VB_DT_DISPATCH_ANY(dtype, (colsum_kernel<kDT><<<grid, 256, 0, st>>>(in, out, rows, cols)));
  VB_LAUNCH_CHECK("colsum_kernel");
  return 0;
}

template <int kDT, int KV>
int launch_ln_bwd_t(cudaStream_t st, const void* dy, const float* x, const float* gamma, float* dx, float* dgamma,
                    float* dbeta, int rows, int dim, float eps, int accumulate, void* dx16, float* dbias_next,
                    const Dropout& drop) {
  const int grid = std::min((rows + 3) / 4, sm_count() * 3);   // persistent: 128-thread blocks, two to three resident per SM
  const size_t smem = 4 * 3 * size_t(dim) * sizeof(float);     // 60 KB at dim 1280
  static PerDevice<bool> configured_on;   // the smem opt-in is per (function, device)
  if (bool& configured = configured_on.here(); !configured) {
    VB_CUDA(cudaFuncSetAttribute(ln_bwd_kernel<kDT, KV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * 3 * 1280 * int(sizeof(float))));
    configured = true;
  }
  ln_bwd_kernel<kDT, KV><<<grid, 128, smem, st>>>(static_cast<const uint16_t*>(dy), x, gamma, dx, dgamma, dbeta, rows, dim, eps,
                                                  accumulate, static_cast<uint16_t*>(dx16), dbias_next, drop);
  VB_LAUNCH_CHECK("ln_bwd_kernel");
  return 0;
}

int launch_ln_bwd(cudaStream_t st, const void* dy, const float* x, const float* gamma, float* dx, float* dgamma,
                  float* dbeta, int rows, int dim, int dtype, float eps, int accumulate, void* dx16, float* dbias_next,
                  const Dropout& drop) {
  if (rows <= 0 || dim <= 0) return fail(VITB200_ERR_INVALID, "ln_bwd: empty problem");
  if (dim & 3) return fail(VITB200_ERR_INVALID, "ln_bwd: dim must be a multiple of 4");
  if (dim > 1280) return fail(VITB200_ERR_UNSUPPORTED, "ln_bwd: dim > 1280 is not built");
#define VB_LN_BWD(KV) VB_DT16_DISPATCH(dtype, return (launch_ln_bwd_t<kDT, KV>(st, dy, x, gamma, dx, dgamma, dbeta, rows, dim, eps, accumulate, dx16, dbias_next, drop)))
  if (dim <= 256) { VB_LN_BWD(2); }
  else if (dim <= 768) { VB_LN_BWD(6); }
  else if (dim <= 1024) { VB_LN_BWD(8); }
  else { VB_LN_BWD(10); }
#undef VB_LN_BWD
  return 0;
}

int launch_pool_ln_bwd(cudaStream_t st, const float* x, float* dpl, const float* gamma, float* dx,
                       float* dgamma, float* dbeta, int batch, int T, int dim, int pool_mean, float eps) {
  if (batch <= 0 || T <= 0 || dim <= 0 || (dim & 3)) return fail(VITB200_ERR_INVALID, "pool_ln_bwd: dim must be a positive multiple of 4");
  const size_t smem = (2 * size_t(dim) + 64) * sizeof(float);
  pool_ln_bwd_kernel<<<batch, 256, smem, st>>>(x, dpl, gamma, dpl, dgamma, dbeta, T, dim, pool_mean, eps);
  VB_LAUNCH_CHECK("pool_ln_bwd_kernel");
  // dx of the whole batch: cls -> row 0 of every image gets the pooled gradient, the others 0; mean -> every row 1/T of it
  const int64_t total4 = int64_t(batch) * T * (dim >> 2);
  pool_scatter_kernel<<<grid_for(total4, 256), 256, 0, st>>>(dpl, dx, total4, T, dim, pool_mean);
  VB_LAUNCH_CHECK("pool_scatter_kernel");
  return 0;
}

int launch_head_bwd(cudaStream_t st, const float* pl, const float* dl, const float* W, float* dW, float* dbias,
                    float* dpl, int batch, int dim, int classes) {
  if (batch <= 0 || dim <= 0 || classes <= 0) return fail(VITB200_ERR_INVALID, "head_bwd: empty problem");
  if (dW) {   // null: no parameter gradients wanted (image-only backward)
    head_wgrad_kernel<<<dim3(unsigned((classes + 255) / 256), unsigned(dim)), 256, 0, st>>>(pl, dl, dW, batch, dim, classes);
    VB_LAUNCH_CHECK("head_wgrad_kernel");
  }
  head_dgrad_kernel<<<unsigned((int64_t(batch) * dim * 32 + 255) / 256), 256, 0, st>>>(dl, W, dpl, batch, dim, classes);
  VB_LAUNCH_CHECK("head_dgrad_kernel");
  if (dbias) {   // dbias[c] += sum_b dl[b, c]  (classes may be odd: one column per thread)
    pos_grad_kernel<<<dim3(unsigned((classes + 255) / 256), 1), 256, 0, st>>>(dl, dbias, batch, 1, classes);
    VB_LAUNCH_CHECK("pos_grad_kernel(head bias)");
  }
  return 0;
}

int launch_token_grads(cudaStream_t st, const float* dx, float* dpos, float* dcls, float* dbias, int batch, int T,
                       int dim, int cls_off) {
  if (batch <= 0 || T <= 0 || dim <= 0) return fail(VITB200_ERR_INVALID, "token_grads: empty problem");
  pos_grad_kernel<<<dim3(unsigned((dim + 255) / 256), unsigned(T)), 256, 0, st>>>(dx, dpos, batch, T, dim);
  VB_LAUNCH_CHECK("pos_grad_kernel");
  cls_bias_grad_kernel<<<dim3(unsigned((dim + 255) / 256), unsigned(std::min(T, 32))), 256, 0, st>>>(dpos, dcls, dbias, T, dim, cls_off);
  VB_LAUNCH_CHECK("cls_bias_grad_kernel");
  return 0;
}

// Adjoint of vit.py:69-79 on tcgen05 (attention_bwd_tc5.cu): resident form up to 208 tokens, streamed form beyond.
// `lse2` = the forward's row log-sum-exp (train_forward keeps it); `workspace` = attention_bwd_workspace_floats floats.
// The per-kernel C entry point has neither: it re-runs the forward kernel into scratch for the log-sum-exp.
bool attention_bwd_needs_workspace(int T) { return !attention_bwd_tc5_supports(T); }

size_t attention_bwd_workspace_floats(int batch, int T, int heads) {
  // D per (image, head, token) [+ beyond 208 tokens: the fp32 dQ accumulator [batch * T, heads * 64]]
  const size_t n = size_t(round_up(int64_t(batch) * heads * T, 64));
  return attention_bwd_needs_workspace(T) ? n + size_t(batch) * T * heads * 64 : n;
}

int launch_attention_bwd(cudaStream_t st, const void* qkv, const void* o_fwd, const void* d_out, void* dqkv, int batch, int T,
                         int heads, int dtype, float* workspace, const float* lse2) {
  if (batch <= 0 || T <= 0 || heads <= 0) return fail(VITB200_ERR_INVALID, "attention_bwd: empty problem");
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(VITB200_ERR_INVALID, "attention_bwd: dtype must be bf16 or fp16");
  const size_t n = size_t(round_up(int64_t(batch) * heads * T, 64));
  const size_t ws_floats = attention_bwd_workspace_floats(batch, T, heads);
  float* ws = workspace;
  float* lse_tmp = nullptr;
  uint16_t* o_tmp = nullptr;
  int rc = 0;
  if (ws == nullptr) VB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_floats * sizeof(float), st));
  if (lse2 == nullptr) {   // per-kernel entry point: the forward kernel again, for its log-sum-exp (its output goes to scratch)
    const size_t o_elems = size_t(batch) * T * heads * 64;
    if (cudaMallocAsync(reinterpret_cast<void**>(&lse_tmp), n * sizeof(float), st) != cudaSuccess ||
        cudaMallocAsync(reinterpret_cast<void**>(&o_tmp), o_elems * sizeof(uint16_t), st) != cudaSuccess)
      rc = fail(VITB200_ERR_CUDA, "attention_bwd: scratch allocation failed");
    if (!rc) rc = launch_attention_tc(st, qkv, o_tmp, batch, T, heads, dtype, lse_tmp);
    lse2 = lse_tmp;
  }
  float* dsum = ws;
  if (!rc) rc = launch_attention_bwd_rowdot(st, d_out, o_fwd, dsum, batch, T, heads, dtype);
  if (!rc) {
    if (attention_bwd_needs_workspace(T))
      rc = launch_attention_bwd_tc5_stream(st, qkv, d_out, dqkv, lse2, dsum, ws + n, batch, T, heads, dtype);
    else
      rc = launch_attention_bwd_tc5(st, qkv, d_out, dqkv, lse2, dsum, batch, T, heads, dtype);
  }
  if (o_tmp) cudaFreeAsync(o_tmp, st);
  if (lse_tmp) cudaFreeAsync(lse_tmp, st);
  if (workspace == nullptr) cudaFreeAsync(ws, st);
  return rc;
}

}  // namespace vb
