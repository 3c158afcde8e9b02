// common.h -- shared host-side declarations for libvitb200 (internal; the public
// surface is include/vitb200.h).
#pragma once
#include <cuda.h>            // CUtensorMap type only; the driver is reached via cudart entry points
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string>

#include "../../include/vitb200.h"
#include "ptx.cuh"   // struct Dropout

namespace vb {

// ---- error plumbing ------------------------------------------------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
void count_launch(int n = 1);
const std::string& last_error_ref();
int64_t launch_count();

#define VB_CUDA(expr)                                              \
  do {                                                             \
    cudaError_t _e = (expr);                                       \
    if (_e != cudaSuccess) return ::vb::cuda_fail(_e, #expr);      \
  } while (0)

#define VB_LAUNCH_CHECK(name)                                      \
  do {                                                             \
    cudaError_t _e = cudaGetLastError();                           \
    if (_e != cudaSuccess) return ::vb::cuda_fail(_e, name);       \
    ::vb::count_launch();                                          \
  } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

int sm_count();   // SMs of the current device (cached per device)
// One value per CUDA device, indexed by the current device: function attributes
// (cudaFuncSetAttribute) and occupancy answers belong to the device they were set / asked on, so a
// process that drives several GPUs must configure each kernel once PER DEVICE.
constexpr int VB_MAX_DEVICES = 64;
template <typename T> struct PerDevice {
  T v[VB_MAX_DEVICES] = {};
  T spill{};            // devices beyond the table are re-configured on every call (correct, just slower)
  T& here() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= VB_MAX_DEVICES) { spill = T{}; return spill; }
    return v[dev];
  }
};
bool pdl_enabled();   // VITB200_PDL=0 turns programmatic dependent launch off (A/B tests)

// cudaLaunchKernelEx with the attributes every kernel of the path uses: programmatic stream
// serialization (the kernel calls pdl_wait() before touching global memory) and, for the tcgen05
// GEMM, a thread-block cluster.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                 cudaStream_t stream, int cluster, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = unsigned(cluster);
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = unsigned(na);
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- TMA descriptors -----------------------------------------------------
// 2-D row-major tensor [rows, cols] (cols contiguous, row pitch = ld elements) of element type
// `dt` (VITB200_DT_*, E4M3 = one byte); box = [box_rows, box_bytes of columns]: 128 bytes with the 128-byte swizzle, or
// 64 bytes with the 64-byte swizzle (dense 64-byte rows in shared memory, 16-byte chunk bits [4,6) ^= address bits [7,9)).
int make_tmap_2d(CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int64_t ld,
                 int box_rows, int dt, int box_bytes = 128);
// 3-D [batch, rows, cols] 16-bit tensor, box = [1, box_rows, 64 cols].
int make_tmap_3d_16(CUtensorMap* out, const void* base, int64_t batch, int64_t rows, int64_t cols,
                    int64_t ld, int box_rows, int dt);

int make_tmap_im2col_patches(CUtensorMap* out, const float* images, int64_t batch, int H, int W, int C, int ph, int pw,
                             int pixels);

// ---- kernels (host launchers; all enqueue on `stream`, return 0 / <0) -----
constexpr int GEMM_BM = 128;   // tcgen05 tile rows (A box rows)
constexpr int GEMM_BN = 256;   // tcgen05 tile cols (Wt box rows)
constexpr int GEMM_BK = 64;

// `dtype` / `out_dtype` are VITB200_DT_* values.
// tmC: output map (16-bit [M,N] box 64 cols for the *_16 epilogues, fp32 [M,N] box 32 cols for
// BIAS_RESID_F32 / BIAS_F32); may be null for PATCH_F32, which stores through `C` directly.
int launch_gemm_tc(cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
                   const CUtensorMap* tmC, const float* bias, void* C, int M, int N, int K,
                   int epilogue, const float* aux, int tokens_per_image, int dtype, int cta_group,
                   const Dropout& drop = Dropout(), int cls_off = 1, const float* cls = nullptr,
                   const LnFold& ln = LnFold(), const float* wscale = nullptr);
// dtype VITB200_DT_E4M3 (the fp8 precision): A [M, K] and Wt [N, K] are E4M3 codes (K-major, k-blocks of 128 elements,
// K % 16 == 0), the accumulator is multiplied by the per-column weight scale `wscale` [N] before the epilogue's own math.
// Epilogues STORE_16 (fp16 out), BIAS_RESID_F32, BIAS_F32 and BIAS_GELU_E4M3 (E4M3 out through a 64-byte-wide map);
// no dropout, no split-K, tile modes 1, 2 and 64.
// LayerNorm fold (gemm_tc.cu header): W' = diag(gamma) W packed to 16-bit [N, Kpad], c[n] = sum_k W'_16[n, k] (of the
// ROUNDED values, so that rstd mean c cancels the mean part of x16 W'_16 exactly), d[n] = sum_k beta[k] W[k, n] (+ bias[n]).
// `scratch`: K * N floats.
int launch_fold_layernorm(cudaStream_t stream, const float* W, const float* gamma, const float* beta, const float* bias,
                          void* Wt, float* c, float* d, int K, int N, int Kpad, int dtype, float* scratch);
// Weight gradient C[M, N] += X[K, M]^T dY[K, N] (fp32 C, TMA reduce-add, split-K `splits`): tmX / tmdY are maps
// over the ROW-MAJOR activations with 64-row x 64-column boxes (MN-major operands, no transposed copies)
int launch_gemm_tc_wgrad(cudaStream_t stream, const CUtensorMap& tmX, const CUtensorMap& tmdY, const CUtensorMap& tmC,
                         const float* zero_bias, float* C, int M, int N, int K, int splits, int dtype, int cta_group);
// `cls` (PATCH epilogue, cls_off == 1): also write the class-token rows b*T = cls + pos[0]
// 1 = one CTA per 128x256 tile (Wt box 256 rows), 2 = CTA pair per 256x256 tile (Wt box 128 rows),
// 4 = cluster of two pairs sharing a multicast weight tile (Wt box 64 rows).
// The Wt tensor map must be encoded with GEMM_BN / cta_group box rows.
int gemm_tc_cta_group(int M);
// tile mode for an [M, N] output: 1, 2, (4) as above or 64 = one CTA per 128x64 tile (Wt box 64 rows)
int gemm_tc_tile_mode(int M, int N);
int launch_gemm_f32(cudaStream_t stream, const float* A, const float* W, const float* bias,
                    float* C, int M, int N, int K, int epilogue, const float* aux,
                    int tokens_per_image, const Dropout& drop = Dropout(), int cls_off = 1);
int launch_layernorm(cudaStream_t stream, const float* x, const float* scale, const float* bias,
                     void* y, int rows, int dim, int out_dtype, float eps = 1e-6f, float* copy = nullptr,
                     int64_t ldx = 0);
// `copy` (training): the kernel also writes x to `copy`, the residual buffer the following GEMM adds into
// `ldx`: row pitch of x in elements (0 = dim); y (and copy) stay dense [rows, dim]
// `lse` (optional): [batch*heads, T] fp32, the row log-sum-exp in the log2 domain, kept for the adjoint and the
// attention maps
// `q_tiles` (> 0): only the first q_tiles 128-query tiles of every (image, head) are computed, the other rows of `out`
// (and of `lse`) are left as they were; 0 = all ceil(T / 128)
int launch_attention_tc(cudaStream_t stream, const void* qkv, void* out, int batch, int T,
                        int heads, int dtype, float* lse = nullptr, int q_tiles = 0);
bool attention_tc5_supports(int T);
int launch_attention_tc5(cudaStream_t stream, const void* qkv, void* out, int batch, int T,
                         int heads, int dtype, float* lse = nullptr, int q_tiles = 0);
// tcgen05 kernel for T > 208: streamed key blocks, online softmax (attention_tc5m.cu)
int launch_attention_tc5m(cudaStream_t stream, const void* qkv, void* out, int batch, int T,
                          int heads, int dtype, float* lse = nullptr, int q_tiles = 0);
int launch_attention_f32(cudaStream_t stream, const float* qkv, float* out, int batch, int T,
                         int heads);
// Attention weights P = exp2(Q K^T sl2 - lse2) of one layer, recomputed on tcgen05 from the to_qkv output and the row
// log-sum-exp of launch_attention_tc (attention_probs_tc5.cu): fp32 element (b, h, i, j) at
// out[b * img_stride + (h * T + i) * T + j], so one launch fills a layer's slice of a [batch, layers, heads, T, T] tensor.
int launch_attention_probs(cudaStream_t stream, const void* qkv, const float* lse2, float* out, int64_t img_stride,
                           int batch, int T, int heads, int dtype);
int launch_patchify(cudaStream_t stream, const float* images, void* patches, int batch, int H,
                    int W, int C, int ph, int pw, int Kpad, int out_dtype, int nchw = 0, int tok_off = 0);
// adjoint of launch_patchify for fp32 patches: images (NHWC, or NCHW) <- patches [batch*(Np+tok_off), Kpad]; every
// pixel written once, the pad columns and the class-token slot rows never read
int launch_unpatchify(cudaStream_t stream, const float* patches, float* images, int batch, int H, int W, int C,
                      int ph, int pw, int Kpad, int nchw = 0, int tok_off = 0);
int launch_cls_rows(cudaStream_t stream, const float* cls, const float* pos, float* x, int batch,
                    int T, int dim, const Dropout& drop = Dropout());
int launch_pool_layernorm(cudaStream_t stream, const float* x, const float* scale,
                          const float* bias, void* y, int batch, int T, int dim, int pool,
                          int out_dtype, float eps = 1e-6f);
int launch_pack_weight(cudaStream_t stream, const float* W, void* Wt, int K, int N, int Kpad,
                       int dtype);
// W fp32 [K, N] (Flax kernel) -> Wt E4M3 [N, Kpad] = satfinite(e4m3(W[k, n] / scale[n])), zero for k >= K, and
// scale[n] = max_k |W[k, n]| / 448 (1 for an all-zero column)
int launch_quantize_weight_e4m3(cudaStream_t stream, const float* W, uint8_t* Wt, float* scale, int K, int N, int Kpad);
// ---- fused patch embedding (patch_tc.cu): im2col TMA + tcgen05 GEMM + cls / pos placement (+ LayerNorm-fold outputs) ----
bool patch_im2col_supported(int pw, int channels, int dim);
// W fp32 [ph*pw*C, D] -> Wt' 16-bit [D, ph*64] (k-block p1 = image row p1 of the patch, padded to 64 columns)
int launch_pack_weight_im2col(cudaStream_t stream, const float* W, void* Wt, int D, int ph, int run, int dtype);
// tmImg: make_tmap_im2col_patches(images, ..., 128 pixels); tmW: 2-D map over Wt' [D, ph*64] with a 256-row box
int launch_patch_embed_im2col(cudaStream_t stream, const CUtensorMap& tmImg, const CUtensorMap& tmW, const float* bias,
                              const float* pos, const float* cls, float* x, int batch, int Np, int gw, int ph, int pw,
                              int channels, int D, int cls_off, int dtype, const LnFold* ln);

// ---- backward pass (backward.cu); 16-bit buffers are of type `dtype` (VITB200_DT_BF16 / _F16) ----
int launch_cast16(cudaStream_t stream, const float* x, void* y, int64_t n, int dtype);
int launch_gelu_fwd(cudaStream_t stream, const void* pre, void* hid, int64_t n, int dtype, const Dropout& drop = Dropout());
int launch_mask_inplace(cudaStream_t stream, float* x, int64_t n, const Dropout& drop);
int launch_gelu_bwd(cudaStream_t stream, const void* pre, const void* dhid, void* dpre, int64_t n, int dtype);
// fused passes: y16 = cast(x), sums[c] += sum_r x[r, c]  /  dpre = dhid * gelu'(pre), sums[c] += sum_r dpre[r, c]
int launch_cast16_colsum(cudaStream_t stream, const float* x, void* y, float* sums, int rows, int cols, int dtype,
                         const Dropout& drop = Dropout());
int launch_gelu_bwd_colsum(cudaStream_t stream, const void* pre, const void* dhid, void* dpre, float* sums, int rows,
                           int cols, int dtype, const Dropout& drop = Dropout());
// out[c, r] = in[r, c], r < rows; zero for rows <= r < rows_pad (the K padding of the wgrad GEMMs)
int launch_transpose16(cudaStream_t stream, const void* in, void* out, int rows, int cols, int rows_pad);
// out[c] += sum_r in[r, c]; dtype may be VITB200_DT_F32
int launch_colsum(cudaStream_t stream, const void* in, float* out, int rows, int cols, int dtype);
// dx (+)= LayerNorm backward of dy (16-bit) at input x; dgamma / dbeta accumulate
int launch_ln_bwd(cudaStream_t stream, const void* dy, const float* x, const float* gamma, float* dx,
                  float* dgamma, float* dbeta, int rows, int dim, int dtype, float eps, int accumulate,
                  void* dx16 = nullptr, float* dbias_next = nullptr, const Dropout& drop = Dropout());
// dx16 / dbias_next / drop: also emit the new dx as 16 bits for the next stage's GEMMs (that stage's dropout mask
// replayed) and add its column sums to that stage's bias gradient
// dpl: in = gradient wrt LayerNorm(pooled), out = gradient wrt pooled (overwritten)
int launch_pool_ln_bwd(cudaStream_t stream, const float* x, float* dpl, const float* gamma, float* dx,
                       float* dgamma, float* dbeta, int batch, int T, int dim, int pool_mean, float eps);
// dW / dbias null: only dpl (the image-only backward)
int launch_head_bwd(cudaStream_t stream, const float* pl, const float* dl, const float* W, float* dW,
                    float* dbias, float* dpl, int batch, int dim, int classes);
int launch_token_grads(cudaStream_t stream, const float* dx, float* dpos, float* dcls, float* dbias, int batch,
                       int T, int dim, int cls_off);
// Adjoint of the fused attention (vit.py:69-79) on tcgen05 (attention_bwd_tc5.cu).  o_fwd: the attention output of the forward
// pass (D = rowsum(dO o O) replaces a full row of dP); lse2: the forward's row log-sum-exp (launch_attention_tc's `lse`; null =
// the forward kernel is run again into scratch for it); workspace: attention_bwd_workspace_floats floats (null = stream-ordered
// scratch allocated per call).  T <= 208: dQ accumulates in TMEM; beyond: in an fp32 buffer of the workspace.
bool attention_bwd_needs_workspace(int T);      // beyond the resident form: the workspace also holds the fp32 dQ accumulator
size_t attention_bwd_workspace_floats(int batch, int T, int heads);
int launch_attention_bwd(cudaStream_t stream, const void* qkv, const void* o_fwd, const void* d_out, void* dqkv,
                         int batch, int T, int heads, int dtype, float* workspace = nullptr, const float* lse2 = nullptr);
bool attention_bwd_tc5_supports(int T);         // the resident form
int launch_attention_bwd_tc5(cudaStream_t stream, const void* qkv, const void* d_out, void* dqkv, const float* lse2,
                             const float* dsum, int batch, int T, int heads, int dtype);
// the same kernel for any T (streamed mode): dQ contributions are summed in dq_acc (fp32 [batch * T, heads * 64]) and
// converted into dqkv at the end
int launch_attention_bwd_tc5_stream(cudaStream_t stream, const void* qkv, const void* d_out, void* dqkv, const float* lse2,
                                    const float* dsum, float* dq_acc, int batch, int T, int heads, int dtype);
int launch_dq_convert(cudaStream_t stream, const float* dq_acc, void* dqkv, int64_t rows, int inner, int dtype);
// dsum [batch*heads, T] = rowsum(dO o O) per (image, head, token): the D of the softmax adjoint
int launch_attention_bwd_rowdot(cudaStream_t stream, const void* d_out, const void* o_fwd, float* dsum, int batch, int T,
                                int heads, int dtype);

// ---- training step (optim.cu) ----
// softmax cross-entropy of logits [B, C] with smoothed one-hot labels: mean loss -> *loss, dscale * dloss/dlogits
int launch_softmax_xent(cudaStream_t stream, const float* logits, const int32_t* labels, int B, int C, float eps,
                        float dscale, float* loss, float* dlogits);
constexpr int OPT_CHUNK = 8192;   // elements of a leaf per CTA of the AdamW kernels
struct OptChunk {                 // one chunk of a trainable leaf: p = leaf + start, off = grad offset of the leaf + start
  float* p;
  int64_t off;                    // into the gradient buffer and mu / nu (same layout)
  int32_t n;                      // elements, <= OPT_CHUNK; a multiple of 4 except in a leaf's last chunk
  int32_t decay;
};
struct OptStatus {                // device-side state of the optimiser, written by the step itself
  float norm;                     // global norm of grad * grad_scale of the last step (NaN: non-finite gradients)
  int32_t count;                  // applied updates (optax's count)
  int32_t skipped;                // the last step was skipped
  int32_t apply;                  // what the update kernel obeys
  float gmul, bc1, bc2;           // grad_scale * clip, 1 - b1^t, 1 - b2^t of the last applied step
};
// global norm (per-chunk partials, then a fixed-order reduction), the step decision, the fused update: 3 launches
int launch_adamw(cudaStream_t stream, const OptChunk* chunks, int nchunks, const float* grads, float* mu, float* nu,
                 double* partial, OptStatus* status, const vitb200_adamw& h);

}  // namespace vb
