// optim.cu -- the on-device training step after the backward pass: softmax cross-entropy with its adjoint
// (optax.softmax_cross_entropy with optax.smooth_labels), and AdamW over every parameter leaf in one launch
// (optax.clip_by_global_norm + optax.adamw under optax.apply_if_finite).
//
// The AdamW step is three launches and reads nothing from the host: the global gradient norm as per-chunk
// partial sums, one CTA that reduces them in a fixed order and decides the step (finite? clip factor, bias
// corrections, count), and the fused update.  Each leaf is cut into OPT_CHUNK-element chunks; the chunk table
// (api.cu) lists the chunks of the trainable leaves only, so one launch covers every leaf whatever its size and
// frozen leaves are neither read nor written.
#include <cmath>

#include "common.h"

namespace vb {
namespace {

constexpr int XENT_THREADS = 256;
constexpr int OPT_THREADS = 256;
constexpr int PREP_THREADS = 1024;

__device__ __forceinline__ float warp_max(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// block-wide reduction in a fixed order (lane tree, then the warp partials in index order)
template <bool MAX>
__device__ float block_reduce(float v, float* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = MAX ? warp_max(v) : warp_sum(v);
  __syncthreads();                  // sh may still be read by a previous call
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  float r = sh[0];
  for (int w = 1; w < nw; ++w) r = MAX ? fmaxf(r, sh[w]) : r + sh[w];
  return r;
}

// One CTA per row b of logits [B, C]: q = (1 - eps) onehot(y_b) + eps / C,
// row_loss[b] = sum_c q_c (lse - z_c) = (1 - eps)((m - z_y) + log s) + eps (log s + mean_c(m - z_c)),
// dlogits[b, c] = dscale (softmax(z)_c - q_c) / B.  Written from the max-subtracted terms so that logits of
// magnitude 1e4 lose nothing to cancellation.  A label outside [0, C) makes the row NaN (loss and dlogits).
__global__ void __launch_bounds__(XENT_THREADS) xent_rows_kernel(const float* __restrict__ logits,
                                                                 const int32_t* __restrict__ labels, int C, float eps,
                                                                 float dscale_over_b, float* __restrict__ dlogits,
                                                                 float* __restrict__ row_loss) {
  __shared__ float sh[XENT_THREADS / 32];
  const int b = blockIdx.x;
  const float* z = logits + int64_t(b) * C;
  float* dz = dlogits + int64_t(b) * C;
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < C; c += blockDim.x) mx = fmaxf(mx, z[c]);
  const float m = block_reduce<true>(mx, sh);
  float se = 0.f, sd = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float d = m - z[c];
    se += expf(-d);
    sd += d;
  }
  const float s = block_reduce<false>(se, sh);
  const float sum_d = block_reduce<false>(sd, sh);
  const int y = labels[b];
  const bool valid = y >= 0 && y < C;
  const float log_s = logf(s), inv_s = 1.f / s, off = eps / float(C);
  if (threadIdx.x == 0) {
    const float l = (1.f - eps) * ((m - z[valid ? y : 0]) + log_s) + eps * (log_s + sum_d / float(C));
    row_loss[b] = valid ? l : __int_as_float(0x7fc00000);
  }
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float p = expf(z[c] - m) * inv_s;
    const float q = (c == y ? 1.f - eps : 0.f) + off;
    dz[c] = valid ? dscale_over_b * (p - q) : __int_as_float(0x7fc00000);
  }
}

// loss = (1/B) sum_b row_loss[b], summed in a fixed order (double) whatever the order the rows finished in
__global__ void __launch_bounds__(OPT_THREADS) xent_mean_kernel(const float* __restrict__ row_loss, int B,
                                                                float* __restrict__ loss) {
  __shared__ double sh[OPT_THREADS];
  double s = 0.0;
  for (int i = threadIdx.x; i < B; i += blockDim.x) s += double(row_loss[i]);
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = blockDim.x / 2; w > 0; w >>= 1) {
    if (int(threadIdx.x) < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) *loss = float(sh[0] / double(B));
}

// ---- AdamW ----------------------------------------------------------------------------------------------------------
// stage 1: partial[k] = sum over chunk k of (g * grad_scale)^2, or NaN when the chunk holds a non-finite gradient
// (tracked per element, so a huge but finite gradient whose square overflows is still "finite", as in optax)
__global__ void __launch_bounds__(OPT_THREADS) sumsq_kernel(const OptChunk* __restrict__ chunks,
                                                            const float* __restrict__ grads, float grad_scale,
                                                            double* __restrict__ partial) {
  __shared__ double sh[OPT_THREADS];
  const OptChunk ch = chunks[blockIdx.x];
  const float* g = grads + ch.off;
  float s = 0.f;
  bool bad = false;
  const int n4 = ch.n >> 2;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(g)[i];
    const float a = v.x * grad_scale, b = v.y * grad_scale, c = v.z * grad_scale, d = v.w * grad_scale;
    bad |= !(isfinite(a) && isfinite(b) && isfinite(c) && isfinite(d));
    s += a * a + b * b + c * c + d * d;
  }
  for (int i = 4 * n4 + threadIdx.x; i < ch.n; i += blockDim.x) {
    const float a = g[i] * grad_scale;
    bad |= !isfinite(a);
    s += a * a;
  }
  bad = __syncthreads_or(bad);
  sh[threadIdx.x] = double(s);
  __syncthreads();
  for (int w = blockDim.x / 2; w > 0; w >>= 1) {
    if (int(threadIdx.x) < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = bad ? __longlong_as_double(0x7ff8000000000000ll) : sh[0];
}

// stage 2 (one CTA): the global norm in a fixed order, the finite verdict, and everything the update reads.  The step
// count lives on the device and advances here only when the step applies, so nothing waits for the host.
__global__ void __launch_bounds__(PREP_THREADS) adamw_prepare_kernel(const double* __restrict__ partial, int nparts,
                                                                     OptStatus* __restrict__ st, float grad_scale,
                                                                     float max_norm, float b1, float b2) {
  __shared__ double sh[PREP_THREADS];
  double s = 0.0;
  bool bad = false;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
    const double v = partial[i];
    if (isnan(v)) bad = true;
    else s += v;
  }
  bad = __syncthreads_or(bad);
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = blockDim.x / 2; w > 0; w >>= 1) {
    if (int(threadIdx.x) < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const double norm = sqrt(sh[0]);
  st->norm = bad ? __int_as_float(0x7fc00000) : float(norm);
  if (bad) {
    st->apply = 0;
    st->skipped = 1;
    return;
  }
  const int t = st->count + 1;
  const double clip = max_norm > 0.f ? double(max_norm) / fmax(norm, double(max_norm)) : 1.0;
  st->gmul = float(double(grad_scale) * clip);
  st->bc1 = float(1.0 - pow(double(b1), double(t)));
  st->bc2 = float(1.0 - pow(double(b2), double(t)));
  st->count = t;
  st->apply = 1;
  st->skipped = 0;
}

struct AdamWArgs {
  float lr, b1, b2, one_minus_b1, one_minus_b2, eps, wd;
};

__device__ __forceinline__ void adamw_elem(float& p, float& mu, float& nu, float graw, float gmul, float bc1, float bc2,
                                           const AdamWArgs& a, float wd) {
  const float g = graw * gmul;
  mu = a.b1 * mu + a.one_minus_b1 * g;
  nu = a.b2 * nu + a.one_minus_b2 * (g * g);
  const float u = (mu / bc1) / (sqrtf(nu / bc2) + a.eps) + wd * p;
  p = p - a.lr * u;
}

// stage 3: p, mu, nu of every chunk, float4 loads and stores with a scalar tail; nothing is written when the step is
// skipped (non-finite gradients): p, mu, nu and count stay bit for bit what they were
__global__ void __launch_bounds__(OPT_THREADS) adamw_update_kernel(const OptChunk* __restrict__ chunks,
                                                                   const float* __restrict__ grads, float* __restrict__ mu,
                                                                   float* __restrict__ nu, const OptStatus* __restrict__ st,
                                                                   AdamWArgs a) {
  if (!st->apply) return;
  const float gmul = st->gmul, bc1 = st->bc1, bc2 = st->bc2;
  const OptChunk ch = chunks[blockIdx.x];
  const float wd = ch.decay ? a.wd : 0.f;
  float* p = ch.p;
  const float* g = grads + ch.off;
  float* m = mu + ch.off;
  float* v = nu + ch.off;
  const int n4 = ch.n >> 2;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    float4 P = reinterpret_cast<float4*>(p)[i], M = reinterpret_cast<float4*>(m)[i], V = reinterpret_cast<float4*>(v)[i];
    const float4 G = reinterpret_cast<const float4*>(g)[i];
    adamw_elem(P.x, M.x, V.x, G.x, gmul, bc1, bc2, a, wd);
    adamw_elem(P.y, M.y, V.y, G.y, gmul, bc1, bc2, a, wd);
    adamw_elem(P.z, M.z, V.z, G.z, gmul, bc1, bc2, a, wd);
    adamw_elem(P.w, M.w, V.w, G.w, gmul, bc1, bc2, a, wd);
    reinterpret_cast<float4*>(p)[i] = P;
    reinterpret_cast<float4*>(m)[i] = M;
    reinterpret_cast<float4*>(v)[i] = V;
  }
  for (int i = 4 * n4 + threadIdx.x; i < ch.n; i += blockDim.x) adamw_elem(p[i], m[i], v[i], g[i], gmul, bc1, bc2, a, wd);
}

}  // namespace

int launch_softmax_xent(cudaStream_t st, const float* logits, const int32_t* labels, int B, int C, float eps, float dscale,
                        float* loss, float* dlogits) {
  float* rows = nullptr;
  VB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&rows), size_t(B) * sizeof(float), st));
  xent_rows_kernel<<<B, XENT_THREADS, 0, st>>>(logits, labels, C, eps, dscale / float(B), dlogits, rows);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) {
    count_launch();
    xent_mean_kernel<<<1, OPT_THREADS, 0, st>>>(rows, B, loss);
    e = cudaGetLastError();
    if (e == cudaSuccess) count_launch();
  }
  cudaFreeAsync(rows, st);
  return e == cudaSuccess ? 0 : cuda_fail(e, "softmax_xent");
}

int launch_adamw(cudaStream_t st, const OptChunk* chunks, int nchunks, const float* grads, float* mu, float* nu,
                 double* partial, OptStatus* status, const vitb200_adamw& h) {
  if (nchunks > 0) {
    sumsq_kernel<<<nchunks, OPT_THREADS, 0, st>>>(chunks, grads, h.grad_scale, partial);
    VB_LAUNCH_CHECK("adamw: sumsq_kernel");
  }
  adamw_prepare_kernel<<<1, PREP_THREADS, 0, st>>>(partial, nchunks, status, h.grad_scale, h.max_grad_norm, h.b1, h.b2);
  VB_LAUNCH_CHECK("adamw: adamw_prepare_kernel");
  if (nchunks > 0) {
    const AdamWArgs a{h.lr, h.b1, h.b2, 1.f - h.b1, 1.f - h.b2, h.eps, h.weight_decay};
    adamw_update_kernel<<<nchunks, OPT_THREADS, 0, st>>>(chunks, grads, mu, nu, status, a);
    VB_LAUNCH_CHECK("adamw: adamw_update_kernel");
  }
  return 0;
}

}  // namespace vb
