// api.cu -- the C ABI of include/vitb200.h: model handle, parameter registry
// (the Flax pytree of vit.py, looked up by path), weight packing, the forward
// schedule of ViT.__call__ (vit.py:127-167) and the per-kernel entry points.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include <cuda_fp16.h>

#include "common.h"

namespace vb {
namespace {

constexpr int DIM_HEAD = 64;   // vit.py:123

struct Leaf {
  std::string path;
  std::vector<int64_t> shape;
  float* dev = nullptr;        // fp32 copy on device
  bool set = false;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

// One Dense layer as the kernels want it.
struct DenseW {
  int leaf_kernel = -1, leaf_bias = -1;   // indices into leaves
  int K = 0, N = 0, Kpad = 0;
  uint16_t* wt = nullptr;                 // bf16/fp16 [N, Kpad] (tensor-core modes)
  uint16_t* wf = nullptr;                 // bf16/fp16 [K, N], the Flax layout: the "W^T" operand of dX = dY W^T (backward only)
  uint8_t* w8 = nullptr;                  // fp8 precision (to_qkv, FeedForward): E4M3 [N, Kpad] instead of wt; tm* map it
  float* wscale = nullptr;                // and its per-column scales [N]
  CUtensorMap tm{};                       // box 256 x 64 over wt (one CTA per tile)
  CUtensorMap tm2{};                      // box 128 x 64 over wt (CTA pair per tile)
  CUtensorMap tm4{};                      // box 64 x 64 over wt (cluster of two pairs, multicast)
  const CUtensorMap& map(int mode) const { return (mode == 4 || mode == 64) ? tm4 : (mode == 2 ? tm2 : tm); }
  // LayerNorm fold (the Dense behind a PreNorm: to_qkv, FeedForward Dense_0): W' = diag(gamma) W packed like wt,
  // c = column sums of the rounded W', d = beta^T W (+ bias)   (gemm_tc.cu header)
  uint16_t* wt_ln = nullptr;
  float* ln_c = nullptr;
  float* ln_d = nullptr;
  CUtensorMap tm_ln{}, tm2_ln{}, tm4_ln{};
  const CUtensorMap& map_ln(int mode) const { return (mode == 4 || mode == 64) ? tm4_ln : (mode == 2 ? tm2_ln : tm_ln); }
};

struct Layer {
  int ln1_scale, ln1_bias, ln2_scale, ln2_bias;
  DenseW qkv, out, ff1, ff2;
};

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }     // the training state (vectors of these) frees itself with the model
  int alloc(size_t count) {
    release();
    if (count == 0) return 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(workspace)");
    n = count;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

struct ActMaps {   // TMA descriptors over the activation workspace for one batch size
  CUtensorMap patches, xn, o, h, pooled;   // A operands
  CUtensorMap c_qkv, c_hid, c_x;           // GEMM outputs (TMA store / reduce-add)
  CUtensorMap xn8, h8, c_hid8;             // fp8: the E4M3 views of xn_h / hid_h (A operands, FF Dense_0 output)
  CUtensorMap o_cls, c_x_cls;              // class-token tail: rows b*T of o_h [B, I] and of x [B, D] (row pitch T*I, T*D)
};

}  // namespace
}  // namespace vb

using namespace vb;

struct vitb200_model {
  vitb200_config cfg{};
  int device = 0;
  int Np = 0, T = 0, K0 = 0, K0pad = 0, inner = 0;
  int cls_off = 1;         // 1: class token in front of every image (vit.py:151-152); 0: SimpleViT
  int nchw = 0;
  float eps = 1e-6f;
  bool project_out = true;
  bool tc = true;          // tensor-core (16-bit operand) path, else fp32 SIMT path
  int dt = VITB200_DT_BF16; // operand type of the tensor-core path
  bool finalized = false;
  bool head_tc = false;
  bool fold = false;          // LayerNorm folded into the GEMMs around it (inference forward, dropout rates 0)
  bool fp8 = false;           // VITB200_PREC_FP8: E4M3 to_qkv / FeedForward GEMMs on the LayerNorm-kernel schedule (dt = fp16)
  bool im2col = false;        // patch embedding as one im2col-TMA + tcgen05 kernel (patch_tc.cu), else patchify + TOKENS GEMM
  uint16_t* patch_wt_i2c = nullptr;   // Wt' [dim, ph*64] for that kernel
  CUtensorMap patch_tm_i2c{};
  std::map<std::pair<const float*, int>, CUtensorMap> img_maps;   // im2col maps by (images pointer, batch)
  uint64_t dropout_key = 0;   // 'dropout' rng stream (vitb200_set_dropout_key)
  uint64_t weights_version = 0;   // bumped by every vitb200_adamw_step: a backward must follow a forward on the same weights
  std::vector<uint8_t> leaf_flags;   // VITB200_LEAF_* per leaf (vitb200_set_leaf_flags)
  bool opt_table_dirty = true;       // the AdamW chunk table must be rebuilt from leaf_flags

  // the Dropout instance `site` of this model (rate 0 => off)
  Dropout drop(float rate, uint32_t site) const {
    Dropout d;
    if (rate > 0.f) {
      d.key_lo = uint32_t(dropout_key);
      d.key_hi = uint32_t(dropout_key >> 32);
      d.site = site;
      const double t = double(rate) * 4294967296.0;
      d.threshold = t >= 4294967295.0 ? 0xFFFFFFFFu : uint32_t(t);
      d.inv_keep = 1.0f / (1.0f - rate);
    }
    return d;
  }

  std::vector<Leaf> leaves;
  std::map<std::string, int> index;
  int leaf_pos = -1, leaf_cls = -1, leaf_head_scale = -1, leaf_head_bias = -1;
  DenseW patch, head;
  std::vector<Layer> layers;

  // activation workspace (bf16 mode uses the bf16 buffers, fp32 mode the f32 ones)
  DevBuf<float> x;                                   // residual stream [B*T, D] fp32 (both modes)
  DevBuf<uint16_t> patches_h, xn_h, qkv_h, o_h, hid_h, pooled_h;
  DevBuf<float> patches_f, xn_f, qkv_f, o_f, hid_f, pooled_f;
  DevBuf<float> stats_a, stats_b;                    // LayerNorm fold: per-row partial (sum, sum sq) of x for LN1 / LN2
  int stats_slots_cap = 0;                           // float pairs per row the two buffers hold
  DevBuf<float> img_stage, logit_stage;              // forward_host staging
  DevBuf<float> attn_lse;                            // attention row log-sum-exp [max_batch*heads, T] of a recording
                                                     // forward (vitb200_forward_attn), allocated by the first one
  bool tokens_partial = false;                       // the last inference forward ran the class-token tail: only rows
                                                     // b*T of x hold the output of the last block (vitb200_debug_tokens)
  // submit_host / wait_host: two jobs in flight (H2D of job k+1 overlaps the forward of job k)
  struct HostJob {
    DevBuf<float> img, logit;
    cudaEvent_t h2d_done = nullptr, fwd_done = nullptr, d2h_done = nullptr;
    bool pending = false;       // submitted, not yet waited for
    bool used = false;          // events have been recorded at least once
  } job[2];
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  int64_t jobs_submitted = 0, jobs_waited = 0;
  std::map<int, ActMaps> act_maps;
  std::vector<std::pair<int, cudaEvent_t>>* prof = nullptr;   // per-launch marks while profiling

  // CUDA graphs of the forward for launch-bound problem sizes (small batches): one instantiated graph
  // per (batch, images pointer, logits pointer), a few per batch size, replayed with one cudaGraphLaunch
  struct FwdGraph {
    const float* images = nullptr;
    float* logits = nullptr;
    cudaGraphExec_t exec = nullptr;
    uint64_t last_use = 0;
  };
  struct GraphSlot {
    std::vector<FwdGraph> entries;
    int captures = 0;          // a caller that never repeats its buffers stops being captured
  };
  std::map<int, GraphSlot> graphs;
  cudaStream_t capture_stream = nullptr;
  uint64_t graph_clock = 0;

  // training (train_forward / backward): activations kept per layer, gradient workspace, leaf gradients
  struct TrainLayer {
    DevBuf<uint16_t> xn1, qkv, o, xn2, pre;   // pre: [2 * rows_cap, mlp] -- FF pre-activation, then its GELU (hid)
    DevBuf<float> lse;                        // attention row log-sum-exp [batch*heads, T] (for the tcgen05 adjoint)
    uint16_t* hid = nullptr;
  };
  struct TrainState {
    int fwd_batch = 0;                    // batch of the last train_forward (0 = none to differentiate)
    bool stale = false;                   // that forward's workspace was overwritten by an inference forward since
    int rows_cap = 0;                     // max_batch * T rounded up to the GEMM tile height (256)
    uint64_t fwd_key = 0;                 // 'dropout' rng key of that forward: the backward replays its masks
    std::vector<DevBuf<float>> xs;        // residual stream before every LayerNorm + after the last layer
    std::vector<TrainLayer> layers;
    DevBuf<float> dx, pooled_ln, dpl, zeros, grads, attn_ws;
    DevBuf<uint16_t> dy16, dhid16, dxn16, do16, dqkv16, tA, tB;
    DevBuf<float> dpatches;               // [rows, K0pad] patch-feature gradient (first image-gradient backward)
    std::vector<size_t> grad_off;         // per leaf: element offset into grads
    bool grads_valid = true;              // false after a backward that did not compute parameter gradients
    bool grads_fresh = false;             // grads hold a parameter backward no optimiser step has consumed yet
    uint64_t fwd_version = 0;             // weights_version of the last train_forward
    // AdamW (allocated by the first step or vitb200_optim_state): moments in the layout of grads, the chunk table of the
    // trainable leaves, the norm partials, the device-side status, the LayerNorm-fold scratch of the weight refresh
    DevBuf<float> mu, nu, fold_scratch;
    DevBuf<double> partial;
    DevBuf<OptChunk> chunks;
    std::vector<OptChunk> chunks_host;
    DevBuf<OptStatus> status;
  };
  std::unique_ptr<TrainState> train;

  ~vitb200_model() {
    for (auto& l : leaves)
      if (l.dev) cudaFree(l.dev);
    auto free_dense = [](DenseW& d) {
      if (d.wt) cudaFree(d.wt);
      if (d.wf) cudaFree(d.wf);
      if (d.w8) cudaFree(d.w8);
      if (d.wscale) cudaFree(d.wscale);
      d.w8 = nullptr;
      d.wscale = nullptr;
      if (d.wt_ln) cudaFree(d.wt_ln);
      if (d.ln_c) cudaFree(d.ln_c);
      if (d.ln_d) cudaFree(d.ln_d);
      d.wt = d.wf = d.wt_ln = nullptr;
      d.ln_c = d.ln_d = nullptr;
    };
    free_dense(patch);
    free_dense(head);
    if (patch_wt_i2c) cudaFree(patch_wt_i2c);
    for (auto& L : layers) { free_dense(L.qkv); free_dense(L.out); free_dense(L.ff1); free_dense(L.ff2); }
    for (auto& g : graphs)
      for (auto& e : g.second.entries)
        if (e.exec) cudaGraphExecDestroy(e.exec);
    if (capture_stream) cudaStreamDestroy(capture_stream);
    x.release();
    patches_h.release(); xn_h.release(); qkv_h.release(); o_h.release(); hid_h.release(); pooled_h.release();
    patches_f.release(); xn_f.release(); qkv_f.release(); o_f.release(); hid_f.release(); pooled_f.release();
    img_stage.release(); logit_stage.release(); attn_lse.release();
    for (auto& j : job) {
      j.img.release(); j.logit.release();
      if (j.h2d_done) cudaEventDestroy(j.h2d_done);
      if (j.fwd_done) cudaEventDestroy(j.fwd_done);
      if (j.d2h_done) cudaEventDestroy(j.d2h_done);
    }
    if (h2d_stream) cudaStreamDestroy(h2d_stream);
    if (d2h_stream) cudaStreamDestroy(d2h_stream);
  }
};

namespace vb_api {

int add_leaf(vitb200_model* m, const std::string& path, std::vector<int64_t> shape) {
  Leaf l;
  l.path = path;
  l.shape = std::move(shape);
  m->leaves.push_back(std::move(l));
  m->index[path] = int(m->leaves.size()) - 1;
  return int(m->leaves.size()) - 1;
}

DenseW add_dense(vitb200_model* m, const std::string& prefix, int K, int N, bool bias) {
  DenseW d;
  d.K = K;
  d.N = N;
  d.Kpad = int(round_up(K, GEMM_BK));
  d.leaf_kernel = add_leaf(m, prefix + "/kernel", {K, N});
  if (bias) d.leaf_bias = add_leaf(m, prefix + "/bias", {N});
  return d;
}

// The params pytree of `ViT` (flax compact auto-naming; SURVEY.md section 8c).
void build_registry(vitb200_model* m) {
  const auto& c = m->cfg;
  const int D = c.dim, I = m->inner;
  m->leaf_pos = add_leaf(m, "pos_embedding", {1, m->T, D});          // vit.py:142
  m->leaf_cls = add_leaf(m, "cls", {1, 1, D});                       // vit.py:144
  m->patch = add_dense(m, "Dense_0", m->K0, D, true);                // vit.py:147
  m->layers.resize(c.depth);
  for (int l = 0; l < c.depth; ++l) {                                // vit.py:102-106
    Layer& L = m->layers[l];
    const std::string tp = "Transformer_0/";
    const std::string att = tp + "Attention_" + std::to_string(l);
    L.qkv = add_dense(m, att + "/Dense_0", D, 3 * I, false);         // vit.py:68
    if (m->project_out) L.out = add_dense(m, att + "/Dense_1", I, D, true);   // vit.py:82
    const std::string ff = tp + "FeedForward_" + std::to_string(l);
    L.ff1 = add_dense(m, ff + "/Dense_0", D, c.mlp_dim, true);       // vit.py:48
    L.ff2 = add_dense(m, ff + "/Dense_1", c.mlp_dim, D, true);       // vit.py:51
    const std::string p1 = tp + "PreNorm_" + std::to_string(2 * l) + "/LayerNorm_0";
    const std::string p2 = tp + "PreNorm_" + std::to_string(2 * l + 1) + "/LayerNorm_0";
    L.ln1_scale = add_leaf(m, p1 + "/scale", {D});                   // vit.py:31
    L.ln1_bias = add_leaf(m, p1 + "/bias", {D});
    L.ln2_scale = add_leaf(m, p2 + "/scale", {D});
    L.ln2_bias = add_leaf(m, p2 + "/bias", {D});
  }
  m->leaf_head_scale = add_leaf(m, "LayerNorm_0/scale", {D});        // vit.py:163
  m->leaf_head_bias = add_leaf(m, "LayerNorm_0/bias", {D});
  m->head = add_dense(m, "Dense_1", D, c.num_classes, true);         // vit.py:165
}

int alloc_workspace(vitb200_model* m) {
  const auto& c = m->cfg;
  const size_t B = size_t(c.max_batch);
  const size_t R = B * m->T, Rp = B * m->Np;
  int rc;
  if ((rc = m->x.alloc(R * c.dim))) return rc;
  if (m->tc) {
    // token layout: one row per token, the class-token slot in front of every image never written
    // by patchify and never used as data by the TOKENS epilogue; zeroed once so the MMA reads defined bits
    if ((rc = m->patches_h.alloc(R * m->K0pad))) return rc;
    VB_CUDA(cudaMemset(m->patches_h.p, 0, R * m->K0pad * sizeof(uint16_t)));
    if ((rc = m->xn_h.alloc(R * c.dim))) return rc;
    if ((rc = m->qkv_h.alloc(R * 3 * m->inner))) return rc;
    if ((rc = m->o_h.alloc(R * m->inner))) return rc;
    if ((rc = m->hid_h.alloc(R * c.mlp_dim))) return rc;
    if (m->fold) {   // slots: 2 per n-tile of a [R, dim] GEMM; the 64-column tiles of small batches need the most
      m->stats_slots_cap = 2 * ceil_div(c.dim, 64);
      if ((rc = m->stats_a.alloc(R * 2 * size_t(m->stats_slots_cap))) || (rc = m->stats_b.alloc(R * 2 * size_t(m->stats_slots_cap)))) return rc;
    }
    if (m->head_tc) { if ((rc = m->pooled_h.alloc(B * c.dim))) return rc; }
    else { if ((rc = m->pooled_f.alloc(B * c.dim))) return rc; }
  } else {
    if ((rc = m->patches_f.alloc(Rp * m->K0pad))) return rc;
    if ((rc = m->xn_f.alloc(R * c.dim))) return rc;
    if ((rc = m->qkv_f.alloc(R * 3 * m->inner))) return rc;
    if ((rc = m->o_f.alloc(R * m->inner))) return rc;
    if ((rc = m->hid_f.alloc(R * c.mlp_dim))) return rc;
    if ((rc = m->pooled_f.alloc(B * c.dim))) return rc;
  }
  return 0;
}

int get_act_maps(vitb200_model* m, int batch, const ActMaps** out) {
  auto it = m->act_maps.find(batch);
  if (it == m->act_maps.end()) {
    const auto& c = m->cfg;
    const int64_t R = int64_t(batch) * m->T;
    ActMaps am;
    int rc;
    const int dt = m->dt;
    if ((rc = make_tmap_2d(&am.patches, m->patches_h.p, R, m->K0pad, m->K0pad, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.xn, m->xn_h.p, R, c.dim, c.dim, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.o, m->o_h.p, R, m->inner, m->inner, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.h, m->hid_h.p, R, c.mlp_dim, c.mlp_dim, GEMM_BM, dt))) return rc;
    if (m->head_tc)
      if ((rc = make_tmap_2d(&am.pooled, m->pooled_h.p, batch, c.dim, c.dim, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.c_qkv, m->qkv_h.p, R, 3 * m->inner, 3 * m->inner, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.c_hid, m->hid_h.p, R, c.mlp_dim, c.mlp_dim, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.c_x, m->x.p, R, c.dim, c.dim, GEMM_BM, VITB200_DT_F32))) return rc;
    const int64_t T = m->T;
    if ((rc = make_tmap_2d(&am.o_cls, m->o_h.p, batch, m->inner, T * m->inner, GEMM_BM, dt))) return rc;
    if ((rc = make_tmap_2d(&am.c_x_cls, m->x.p, batch, c.dim, T * c.dim, GEMM_BM, VITB200_DT_F32))) return rc;
    if (m->fp8) {   // E4M3 codes in the first half of the 16-bit buffers' bytes: the workspace does not grow
      if ((rc = make_tmap_2d(&am.xn8, m->xn_h.p, R, c.dim, c.dim, GEMM_BM, VITB200_DT_E4M3))) return rc;
      if ((rc = make_tmap_2d(&am.h8, m->hid_h.p, R, c.mlp_dim, c.mlp_dim, GEMM_BM, VITB200_DT_E4M3))) return rc;
      if ((rc = make_tmap_2d(&am.c_hid8, m->hid_h.p, R, c.mlp_dim, c.mlp_dim, GEMM_BM, VITB200_DT_E4M3, 64))) return rc;
    }
    it = m->act_maps.emplace(batch, am).first;
  }
  *out = &it->second;
  return 0;
}

// the 16-bit copies of one Dense kernel re-derived from its fp32 leaf, into the buffers they already have
int repack_dense(vitb200_model* m, DenseW& d, cudaStream_t st) {
  if (d.leaf_kernel < 0) return 0;
  int rc = launch_pack_weight(st, m->leaves[d.leaf_kernel].dev, d.wt, d.K, d.N, d.Kpad, m->dt);
  if (rc) return rc;
  if (d.wf && (rc = launch_cast16(st, m->leaves[d.leaf_kernel].dev, d.wf, int64_t(d.K) * d.N, m->dt))) return rc;
  return 0;
}

int pack_dense(vitb200_model* m, DenseW& d, cudaStream_t st) {
  if (d.leaf_kernel < 0) return 0;
  if (d.wt == nullptr)
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.wt), size_t(d.N) * d.Kpad * sizeof(uint16_t)));
  int rc = repack_dense(m, d, st);
  if (rc) return rc;
  if ((rc = make_tmap_2d(&d.tm, d.wt, d.N, d.Kpad, d.Kpad, GEMM_BN, m->dt))) return rc;
  if ((rc = make_tmap_2d(&d.tm2, d.wt, d.N, d.Kpad, d.Kpad, GEMM_BN / 2, m->dt))) return rc;
  return make_tmap_2d(&d.tm4, d.wt, d.N, d.Kpad, d.Kpad, GEMM_BN / 4, m->dt);
}

// fp8: the Dense as E4M3 codes [N, Kpad] + per-column scales; the tensor maps tm / tm2 / tm4 point at the codes
int quant_dense(vitb200_model* m, DenseW& d, cudaStream_t st) {
  if (d.w8 == nullptr) {
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.w8), size_t(d.N) * d.Kpad));
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.wscale), size_t(d.N) * sizeof(float)));
  }
  int rc = launch_quantize_weight_e4m3(st, m->leaves[d.leaf_kernel].dev, d.w8, d.wscale, d.K, d.N, d.Kpad);
  if (rc) return rc;
  if ((rc = make_tmap_2d(&d.tm, d.w8, d.N, d.Kpad, d.Kpad, GEMM_BN, VITB200_DT_E4M3))) return rc;
  if ((rc = make_tmap_2d(&d.tm2, d.w8, d.N, d.Kpad, d.Kpad, GEMM_BN / 2, VITB200_DT_E4M3))) return rc;
  return make_tmap_2d(&d.tm4, d.w8, d.N, d.Kpad, d.Kpad, GEMM_BN / 4, VITB200_DT_E4M3);
}

inline const float* leaf_ptr(const vitb200_model* m, int idx) { return idx >= 0 ? m->leaves[idx].dev : nullptr; }

// launch_fold_layernorm's K * N scratch for the largest folded Dense (to_qkv or FeedForward Dense_0)
inline size_t fold_scratch_floats(const vitb200_model* m) { return size_t(m->cfg.dim) * std::max(3 * m->inner, m->cfg.mlp_dim); }

// The Dense that follows a PreNorm, with that LayerNorm folded in (gemm_tc.cu header)
int refold_dense(vitb200_model* m, DenseW& d, int ln_scale, int ln_bias, float* scratch, cudaStream_t st) {
  return launch_fold_layernorm(st, m->leaves[d.leaf_kernel].dev, leaf_ptr(m, ln_scale), leaf_ptr(m, ln_bias),
                               leaf_ptr(m, d.leaf_bias), d.wt_ln, d.ln_c, d.ln_d, d.K, d.N, d.Kpad, m->dt, scratch);
}

int fold_dense(vitb200_model* m, DenseW& d, int ln_scale, int ln_bias, float* scratch, cudaStream_t st) {
  if (d.wt_ln == nullptr) {
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.wt_ln), size_t(d.N) * d.Kpad * sizeof(uint16_t)));
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.ln_c), size_t(d.N) * sizeof(float)));
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.ln_d), size_t(d.N) * sizeof(float)));
  }
  int rc = refold_dense(m, d, ln_scale, ln_bias, scratch, st);
  if (rc) return rc;
  if ((rc = make_tmap_2d(&d.tm_ln, d.wt_ln, d.N, d.Kpad, d.Kpad, GEMM_BN, m->dt))) return rc;
  if ((rc = make_tmap_2d(&d.tm2_ln, d.wt_ln, d.N, d.Kpad, d.Kpad, GEMM_BN / 2, m->dt))) return rc;
  return make_tmap_2d(&d.tm4_ln, d.wt_ln, d.N, d.Kpad, d.Kpad, GEMM_BN / 4, m->dt);
}

// profiling marks: one event BEFORE each launch (+ one at the end); launches are back to back
// on one stream, so the gap between consecutive marks is that launch's duration.
inline void mark(vitb200_model* m, cudaStream_t st, int cat) {
  if (!m->prof) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  m->prof->emplace_back(cat, e);
}

__global__ void add_16_into_f32_kernel(const uint16_t* __restrict__ a, float* __restrict__ x, int64_t n, int dt) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i < n) x[i] += dt == VITB200_DT_F16 ? __half2float(__ushort_as_half(a[i])) : __uint_as_float(uint32_t(a[i]) << 16);
}
__global__ void add_f32_into_f32_kernel(const float* __restrict__ a, float* __restrict__ x, int64_t n) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i < n) x[i] += a[i];
}

int forward_head(vitb200_model* m, cudaStream_t st, const ActMaps* am, int batch, float* logits);

// Layers whose attention weights a forward records (vitb200_forward_attn): slot[l] = position of layer l in `maps`
// [batch, n, heads, T, T] fp32, or -1.
struct AttnRecord {
  std::vector<int> slot;
  int n = 0;
  float* maps = nullptr;
};

// The attention of layer l (vit.py:69-79).  A recorded layer also keeps the row log-sum-exp and, while qkv_h still
// holds this layer's q / k, recomputes P = exp2(s sl2 - lse2) into its slice of the maps (attention_probs_tc5.cu); one
// lse buffer serves every layer, the probabilities kernel has consumed it before the next layer's attention runs.
// `q_tiles` as launch_attention_tc: 1 in the class-token tail, which never records.
int attention_layer(vitb200_model* m, cudaStream_t st, int batch, int l, const AttnRecord* rec, int q_tiles = 0) {
  const int T = m->T, heads = m->cfg.heads;
  const int slot = rec ? rec->slot[l] : -1;
  if (slot < 0) return launch_attention_tc(st, m->qkv_h.p, m->o_h.p, batch, T, heads, m->dt, nullptr, q_tiles);
  int rc;
  if ((rc = launch_attention_tc(st, m->qkv_h.p, m->o_h.p, batch, T, heads, m->dt, m->attn_lse.p))) return rc;
  const int64_t per_layer = int64_t(heads) * T * T;
  return launch_attention_probs(st, m->qkv_h.p, m->attn_lse.p, rec->maps + slot * per_layer, rec->n * per_layer, batch, T,
                                heads, m->dt);
}

// vit.py:146-153 as one kernel (patch_tc.cu): im2col TMA over the caller's images + GEMM + cls / pos placement; `ln` non-null
// adds the LayerNorm-fold outputs.  The im2col map depends on the images pointer: kept per (pointer, batch), a handful.
int patch_embed_im2col(vitb200_model* m, cudaStream_t st, const float* images, int batch, const LnFold* ln) {
  const auto& c = m->cfg;
  auto key = std::make_pair(images, batch);
  auto it = m->img_maps.find(key);
  if (it == m->img_maps.end()) {
    if (m->img_maps.size() >= 64) m->img_maps.clear();
    CUtensorMap tm;
    int rc = make_tmap_im2col_patches(&tm, images, batch, c.image_h, c.image_w, c.channels, c.patch_h, c.patch_w, 128);
    if (rc) return rc;
    it = m->img_maps.emplace(key, tm).first;
  }
  return launch_patch_embed_im2col(st, it->second, m->patch_tm_i2c, leaf_ptr(m, m->patch.leaf_bias), leaf_ptr(m, m->leaf_pos),
                                   leaf_ptr(m, m->leaf_cls), m->x.p, batch, m->Np, c.image_w / c.patch_w, c.patch_h, c.patch_w,
                                   c.channels, c.dim, m->cls_off, m->dt, ln);
}

// The class-token tail (DESIGN.md section 3).  With pool = 'cls' the logits read row b*T of the token stream alone, and in
// the last block that row depends on the other rows only through their keys and values: to_qkv runs over every row,
// attention over q tile 0 (which holds the class query) of every (image, head), and to_out, FF Dense_0 and FF Dense_1 as
// GEMMs of M = batch rows over the class-token rows.  Their tile mode and statistics slots stay those of the [B*T, N]
// GEMMs, so the class rows see the same MMA shape and the same summation order: the logits are bit-identical.  Kept off
// where other rows matter or are indexed: mean pooling, dropout (masks by token row), an identity to_out, the fp32 path,
// and a forward that records the last layer's attention weights (every query row; the whole tail then runs in full).
bool cls_tail(const vitb200_model* m, const AttnRecord* rec) {
  const auto& c = m->cfg;
  return m->tc && c.pool == VITB200_POOL_CLS && m->cls_off == 1 && m->project_out && c.depth > 0 && c.dropout == 0.f &&
         c.emb_dropout == 0.f && !(rec && rec->slot[size_t(c.depth - 1)] >= 0);
}

// ---- the forward schedule with every PreNorm LayerNorm folded into the GEMMs around it: 4 + 5L launches ----
// patchify | patch GEMM (TOKENS_LN: x, x16, stats_a) | per layer: to_qkv (LN_STORE_16 on x16 / stats_a) | attention |
// to_out (RESID_LN: x, x16, stats_b) | FF Dense_0 (LN_GELU_16 on x16 / stats_b) | FF Dense_1 (RESID_LN -> stats_a; plain
// RESID in the last layer) | pool + LayerNorm | head.  x16 lives in the buffer the LayerNorm kernel used to write.
// In the class-token tail the last layer's to_out / FF GEMMs write x16, stats_b and hid compact ([batch, ...]); its to_qkv
// has consumed xn_h and stats_a before.
int forward_tc_fold(vitb200_model* m, cudaStream_t st, const float* images, int batch, float* logits,
                    const AttnRecord* rec = nullptr) {
  const auto& c = m->cfg;
  const int D = c.dim, I = m->inner, T = m->T;
  const int R = batch * T;
  const ActMaps* am;
  int rc;
  if ((rc = get_act_maps(m, batch, &am))) return rc;
  const int cg_qkv = gemm_tc_tile_mode(R, 3 * I), cg_d = gemm_tc_tile_mode(R, D), cg_ff1 = gemm_tc_tile_mode(R, c.mlp_dim);
  LnFold out_a, out_b, in_a, in_b;                 // producers write x16 + stats, consumers read stats + c
  out_a.x16 = out_b.x16 = m->xn_h.p;
  out_a.stats = in_a.stats = reinterpret_cast<float2*>(m->stats_a.p);
  out_b.stats = in_b.stats = reinterpret_cast<float2*>(m->stats_b.p);
  out_a.slots = out_b.slots = in_a.slots = in_b.slots = 2 * ceil_div(D, cg_d == 64 ? 64 : GEMM_BN);
  in_a.eps = in_b.eps = m->eps;
  // the im2col kernel's statistics slots are 2 per 256-column tile: usable whenever the other producers use the same count
  if (m->im2col && out_a.slots % (2 * ceil_div(D, GEMM_BN)) == 0 && (reinterpret_cast<uintptr_t>(images) & 15) == 0) {
    mark(m, st, VITB200_CAT_GEMM_PATCH);
    if ((rc = patch_embed_im2col(m, st, images, batch, &out_a))) return rc;
  } else {
    mark(m, st, VITB200_CAT_PATCHIFY);
    if ((rc = launch_patchify(st, images, m->patches_h.p, batch, c.image_h, c.image_w, c.channels,
                              c.patch_h, c.patch_w, m->K0pad, m->dt, m->nchw, m->cls_off))) return rc;
    mark(m, st, VITB200_CAT_GEMM_PATCH);
    if ((rc = launch_gemm_tc(st, am->patches, m->patch.map(cg_d), &am->c_x, leaf_ptr(m, m->patch.leaf_bias), m->x.p,
                             R, D, m->K0pad, VITB200_EPI_TOKENS_LN, leaf_ptr(m, m->leaf_pos), T, m->dt, cg_d,
                             Dropout(), m->cls_off, leaf_ptr(m, m->leaf_cls), out_a))) return rc;
  }
  const bool tail = cls_tail(m, rec);
  for (int l = 0; l < c.depth; ++l) {   // vit.py:108-110
    Layer& L = m->layers[l];
    const bool cls_rows = tail && l + 1 == c.depth;   // rows after attention: the class tokens alone
    const int M = cls_rows ? batch : R;
    const CUtensorMap& a_o = cls_rows ? am->o_cls : am->o;
    const CUtensorMap& c_x = cls_rows ? am->c_x_cls : am->c_x;
    // Residual(PreNorm(Attention))  vit.py:31,39,62-87
    mark(m, st, VITB200_CAT_GEMM_QKV);
    in_a.c = L.qkv.ln_c;
    if ((rc = launch_gemm_tc(st, am->xn, L.qkv.map_ln(cg_qkv), &am->c_qkv, L.qkv.ln_d, m->qkv_h.p, R, 3 * I, D,
                             VITB200_EPI_LN_STORE_16, nullptr, 0, m->dt, cg_qkv, Dropout(), m->cls_off, nullptr, in_a))) return rc;
    mark(m, st, VITB200_CAT_ATTENTION);
    if ((rc = attention_layer(m, st, batch, l, rec, cls_rows ? 1 : 0))) return rc;
    mark(m, st, VITB200_CAT_GEMM_OUT);
    if ((rc = launch_gemm_tc(st, a_o, L.out.map(cg_d), &c_x, leaf_ptr(m, L.out.leaf_bias), m->x.p, M, D, I,
                             VITB200_EPI_RESID_LN, nullptr, 0, m->dt, cg_d, Dropout(), m->cls_off, nullptr, out_b))) return rc;
    // Residual(PreNorm(FeedForward))  vit.py:31,39,47-53
    mark(m, st, VITB200_CAT_GEMM_FF1);
    in_b.c = L.ff1.ln_c;
    if ((rc = launch_gemm_tc(st, am->xn, L.ff1.map_ln(cg_ff1), &am->c_hid, L.ff1.ln_d, m->hid_h.p, M, c.mlp_dim, D,
                             VITB200_EPI_LN_GELU_16, nullptr, 0, m->dt, cg_ff1, Dropout(), m->cls_off, nullptr, in_b))) return rc;
    mark(m, st, VITB200_CAT_GEMM_FF2);
    if (l + 1 < c.depth) {
      if ((rc = launch_gemm_tc(st, am->h, L.ff2.map(cg_d), &am->c_x, leaf_ptr(m, L.ff2.leaf_bias), m->x.p, R, D, c.mlp_dim,
                               VITB200_EPI_RESID_LN, nullptr, 0, m->dt, cg_d, Dropout(), m->cls_off, nullptr, out_a))) return rc;
    } else {   // nothing normalises the last layer's output row by row: pool + head LayerNorm read x itself
      if ((rc = launch_gemm_tc(st, am->h, L.ff2.map(cg_d), &c_x, leaf_ptr(m, L.ff2.leaf_bias), m->x.p, M, D, c.mlp_dim,
                               VITB200_EPI_BIAS_RESID_F32, nullptr, 0, m->dt, cg_d))) return rc;
    }
  }
  return forward_head(m, st, am, batch, logits);
}

// ---- the forward schedule, bf16 / tcgen05 flavour ---------------------------
// `rec` (vitb200_forward_attn): record the attention weights of some layers; null = the plain forward
int forward_tc(vitb200_model* m, cudaStream_t st, const float* images, int batch, float* logits,
               const AttnRecord* rec = nullptr) {
  if (m->fold) return forward_tc_fold(m, st, images, batch, logits, rec);
  const auto& c = m->cfg;
  const int D = c.dim, I = m->inner, T = m->T;
  const int R = batch * T;
  const ActMaps* am;
  int rc;
  if ((rc = get_act_maps(m, batch, &am))) return rc;
  // tile mode per GEMM shape (pairs for anything that fills the machine, small tiles otherwise)
  const int cgp = gemm_tc_tile_mode(R, D);
  const int cg_qkv = gemm_tc_tile_mode(R, 3 * I), cg_d = gemm_tc_tile_mode(R, D), cg_ff1 = gemm_tc_tile_mode(R, c.mlp_dim);
  const int ln_dt = m->fp8 ? VITB200_DT_E4M3 : m->dt;   // the LayerNorm output is the A operand of to_qkv / FF Dense_0
  if (m->im2col && (reinterpret_cast<uintptr_t>(images) & 15) == 0) {
    mark(m, st, VITB200_CAT_GEMM_PATCH);
    if ((rc = patch_embed_im2col(m, st, images, batch, nullptr))) return rc;
  } else {
    // vit.py:146  patchify (+ fp32->16-bit cast, zero pad to K0pad) into the token layout: row b*T+cls+t
    mark(m, st, VITB200_CAT_PATCHIFY);
    if ((rc = launch_patchify(st, images, m->patches_h.p, batch, c.image_h, c.image_w, c.channels,
                              c.patch_h, c.patch_w, m->K0pad, m->dt, m->nchw, m->cls_off))) return rc;
    // vit.py:147-153  Dense_0 + bias + pos_embedding[t] over all B*T token rows; the class-token row of
    // every image (t = 0) is cls + pos_embedding[0], written by the same epilogue
    mark(m, st, VITB200_CAT_GEMM_PATCH);
    if ((rc = launch_gemm_tc(st, am->patches, m->patch.map(cgp), &am->c_x, leaf_ptr(m, m->patch.leaf_bias), m->x.p,
                               R, D, m->K0pad, VITB200_EPI_TOKENS_F32, leaf_ptr(m, m->leaf_pos), T, m->dt, cgp,
                               m->drop(c.emb_dropout, 0), m->cls_off, leaf_ptr(m, m->leaf_cls)))) return rc;
  }
  const bool tail = cls_tail(m, rec);
  for (int l = 0; l < c.depth; ++l) {   // vit.py:108-110
    Layer& L = m->layers[l];
    // class-token tail: after attention the last layer works on rows b*T alone, its second LayerNorm writes xn_h compact
    const bool cls_rows = tail && l + 1 == c.depth;
    const int M = cls_rows ? batch : R;
    const CUtensorMap& a_o = cls_rows ? am->o_cls : am->o;
    const CUtensorMap& c_x = cls_rows ? am->c_x_cls : am->c_x;
    // Residual(PreNorm(Attention))  vit.py:31,39,62-87
    mark(m, st, VITB200_CAT_LAYERNORM);
    if ((rc = launch_layernorm(st, m->x.p, leaf_ptr(m, L.ln1_scale), leaf_ptr(m, L.ln1_bias), m->xn_h.p, R, D, ln_dt, m->eps))) return rc;
    mark(m, st, VITB200_CAT_GEMM_QKV);
    if (m->fp8) {
      if ((rc = launch_gemm_tc(st, am->xn8, L.qkv.map(cg_qkv), &am->c_qkv, nullptr, m->qkv_h.p, R, 3 * I, D, VITB200_EPI_STORE_16,
                               nullptr, 0, VITB200_DT_E4M3, cg_qkv, Dropout(), m->cls_off, nullptr, LnFold(), L.qkv.wscale))) return rc;
    } else if ((rc = launch_gemm_tc(st, am->xn, L.qkv.map(cg_qkv), &am->c_qkv, nullptr, m->qkv_h.p, R, 3 * I, D, VITB200_EPI_STORE_16, nullptr, 0, m->dt, cg_qkv))) return rc;
    mark(m, st, VITB200_CAT_ATTENTION);
    if ((rc = attention_layer(m, st, batch, l, rec, cls_rows ? 1 : 0))) return rc;
    mark(m, st, VITB200_CAT_GEMM_OUT);
    if (m->project_out) {
      if ((rc = launch_gemm_tc(st, a_o, L.out.map(cg_d), &c_x, leaf_ptr(m, L.out.leaf_bias), m->x.p, M, D, I, VITB200_EPI_BIAS_RESID_F32, nullptr, 0, m->dt, cg_d, m->drop(c.dropout, 1 + 3 * l)))) return rc;
    } else {   // heads == 1 and dim == 64: to_out is the identity (vit.py:65,85)
      const int64_t n = int64_t(R) * D;
      add_16_into_f32_kernel<<<unsigned((n + 255) / 256), 256, 0, st>>>(m->o_h.p, m->x.p, n, m->dt);
      VB_LAUNCH_CHECK("add_16_into_f32_kernel");
    }
    // Residual(PreNorm(FeedForward))  vit.py:31,39,47-53
    mark(m, st, VITB200_CAT_LAYERNORM);
    if ((rc = launch_layernorm(st, m->x.p, leaf_ptr(m, L.ln2_scale), leaf_ptr(m, L.ln2_bias), m->xn_h.p, M, D, ln_dt, m->eps,
                               nullptr, cls_rows ? int64_t(T) * D : D))) return rc;
    if (m->fp8) {   // E4M3 in, E4M3 hidden activations, E4M3 in again: FF Dense_0 -> GELU -> FF Dense_1
      mark(m, st, VITB200_CAT_GEMM_FF1);
      if ((rc = launch_gemm_tc(st, am->xn8, L.ff1.map(cg_ff1), &am->c_hid8, leaf_ptr(m, L.ff1.leaf_bias), m->hid_h.p, M, c.mlp_dim, D,
                               VITB200_EPI_BIAS_GELU_E4M3, nullptr, 0, VITB200_DT_E4M3, cg_ff1, Dropout(), m->cls_off, nullptr,
                               LnFold(), L.ff1.wscale))) return rc;
      mark(m, st, VITB200_CAT_GEMM_FF2);
      if ((rc = launch_gemm_tc(st, am->h8, L.ff2.map(cg_d), &c_x, leaf_ptr(m, L.ff2.leaf_bias), m->x.p, M, D, c.mlp_dim,
                               VITB200_EPI_BIAS_RESID_F32, nullptr, 0, VITB200_DT_E4M3, cg_d, Dropout(), m->cls_off, nullptr,
                               LnFold(), L.ff2.wscale))) return rc;
      continue;
    }
    mark(m, st, VITB200_CAT_GEMM_FF1);
    if ((rc = launch_gemm_tc(st, am->xn, L.ff1.map(cg_ff1), &am->c_hid, leaf_ptr(m, L.ff1.leaf_bias), m->hid_h.p, M, c.mlp_dim, D, VITB200_EPI_BIAS_GELU_16, nullptr, 0, m->dt, cg_ff1, m->drop(c.dropout, 2 + 3 * l)))) return rc;
    mark(m, st, VITB200_CAT_GEMM_FF2);
    if ((rc = launch_gemm_tc(st, am->h, L.ff2.map(cg_d), &c_x, leaf_ptr(m, L.ff2.leaf_bias), m->x.p, M, D, c.mlp_dim, VITB200_EPI_BIAS_RESID_F32, nullptr, 0, m->dt, cg_d, m->drop(c.dropout, 3 + 3 * l)))) return rc;
  }
  return forward_head(m, st, am, batch, logits);
}

// vit.py:159-165  pool, LayerNorm_0, Dense_1
int forward_head(vitb200_model* m, cudaStream_t st, const ActMaps* am, int batch, float* logits) {
  const auto& c = m->cfg;
  const int D = c.dim, T = m->T;
  const int cgh = gemm_tc_tile_mode(batch, c.num_classes);
  int rc;
  if (m->head_tc) {
    mark(m, st, VITB200_CAT_POOL_LN);
    if ((rc = launch_pool_layernorm(st, m->x.p, leaf_ptr(m, m->leaf_head_scale), leaf_ptr(m, m->leaf_head_bias), m->pooled_h.p, batch, T, D, c.pool, m->dt, m->eps))) return rc;
    mark(m, st, VITB200_CAT_GEMM_HEAD);
    CUtensorMap c_logits;   // the caller's buffer: encoded per call (host-side, ~1 us)
    if ((rc = make_tmap_2d(&c_logits, logits, batch, c.num_classes, c.num_classes, GEMM_BM, VITB200_DT_F32))) return rc;
    if ((rc = launch_gemm_tc(st, am->pooled, m->head.map(cgh), &c_logits, leaf_ptr(m, m->head.leaf_bias), logits, batch, c.num_classes, D, VITB200_EPI_BIAS_F32, nullptr, 0, m->dt, cgh))) return rc;
  } else {
    mark(m, st, VITB200_CAT_POOL_LN);
    if ((rc = launch_pool_layernorm(st, m->x.p, leaf_ptr(m, m->leaf_head_scale), leaf_ptr(m, m->leaf_head_bias), m->pooled_f.p, batch, T, D, c.pool, VITB200_DT_F32, m->eps))) return rc;
    mark(m, st, VITB200_CAT_GEMM_HEAD);
    if ((rc = launch_gemm_f32(st, m->pooled_f.p, leaf_ptr(m, m->head.leaf_kernel), leaf_ptr(m, m->head.leaf_bias), logits, batch, c.num_classes, D, VITB200_EPI_BIAS_F32, nullptr, 0))) return rc;
  }
  return 0;
}

// ---- the forward schedule, fp32 validation flavour --------------------------
int forward_f32(vitb200_model* m, cudaStream_t st, const float* images, int batch, float* logits) {
  const auto& c = m->cfg;
  const int D = c.dim, I = m->inner, T = m->T, Np = m->Np;
  const int R = batch * T, Rp = batch * Np;
  int rc;
  mark(m, st, VITB200_CAT_PATCHIFY);
  if ((rc = launch_patchify(st, images, m->patches_f.p, batch, c.image_h, c.image_w, c.channels,
                            c.patch_h, c.patch_w, m->K0pad, VITB200_DT_F32, m->nchw))) return rc;
  // fp32 mode keeps K0pad == K0 (checked at create), so the patch matrix is a dense [Rp, K0].
  mark(m, st, VITB200_CAT_GEMM_PATCH);
  if ((rc = launch_gemm_f32(st, m->patches_f.p, leaf_ptr(m, m->patch.leaf_kernel), leaf_ptr(m, m->patch.leaf_bias), m->x.p,
                            Rp, D, m->K0, VITB200_EPI_PATCH_F32, leaf_ptr(m, m->leaf_pos), Np, m->drop(c.emb_dropout, 0), m->cls_off))) return rc;
  mark(m, st, VITB200_CAT_CLS_ROWS);
  if (m->cls_off && (rc = launch_cls_rows(st, leaf_ptr(m, m->leaf_cls), leaf_ptr(m, m->leaf_pos), m->x.p, batch, T, D, m->drop(c.emb_dropout, 0)))) return rc;
  for (int l = 0; l < c.depth; ++l) {
    Layer& L = m->layers[l];
    mark(m, st, VITB200_CAT_LAYERNORM);
    if ((rc = launch_layernorm(st, m->x.p, leaf_ptr(m, L.ln1_scale), leaf_ptr(m, L.ln1_bias), m->xn_f.p, R, D, VITB200_DT_F32, m->eps))) return rc;
    mark(m, st, VITB200_CAT_GEMM_QKV);
    if ((rc = launch_gemm_f32(st, m->xn_f.p, leaf_ptr(m, L.qkv.leaf_kernel), nullptr, m->qkv_f.p, R, 3 * I, D, VITB200_EPI_STORE_16, nullptr, 0))) return rc;
    mark(m, st, VITB200_CAT_ATTENTION);
    if ((rc = launch_attention_f32(st, m->qkv_f.p, m->o_f.p, batch, T, c.heads))) return rc;
    mark(m, st, VITB200_CAT_GEMM_OUT);
    if (m->project_out) {
      if ((rc = launch_gemm_f32(st, m->o_f.p, leaf_ptr(m, L.out.leaf_kernel), leaf_ptr(m, L.out.leaf_bias), m->x.p, R, D, I, VITB200_EPI_BIAS_RESID_F32, nullptr, 0, m->drop(c.dropout, 1 + 3 * l)))) return rc;
    } else {
      const int64_t n = int64_t(R) * D;
      add_f32_into_f32_kernel<<<unsigned((n + 255) / 256), 256, 0, st>>>(m->o_f.p, m->x.p, n);
      VB_LAUNCH_CHECK("add_f32_into_f32_kernel");
    }
    mark(m, st, VITB200_CAT_LAYERNORM);
    if ((rc = launch_layernorm(st, m->x.p, leaf_ptr(m, L.ln2_scale), leaf_ptr(m, L.ln2_bias), m->xn_f.p, R, D, VITB200_DT_F32, m->eps))) return rc;
    mark(m, st, VITB200_CAT_GEMM_FF1);
    if ((rc = launch_gemm_f32(st, m->xn_f.p, leaf_ptr(m, L.ff1.leaf_kernel), leaf_ptr(m, L.ff1.leaf_bias), m->hid_f.p, R, c.mlp_dim, D, VITB200_EPI_BIAS_GELU_16, nullptr, 0, m->drop(c.dropout, 2 + 3 * l)))) return rc;
    mark(m, st, VITB200_CAT_GEMM_FF2);
    if ((rc = launch_gemm_f32(st, m->hid_f.p, leaf_ptr(m, L.ff2.leaf_kernel), leaf_ptr(m, L.ff2.leaf_bias), m->x.p, R, D, c.mlp_dim, VITB200_EPI_BIAS_RESID_F32, nullptr, 0, m->drop(c.dropout, 3 + 3 * l)))) return rc;
  }
  mark(m, st, VITB200_CAT_POOL_LN);
  if ((rc = launch_pool_layernorm(st, m->x.p, leaf_ptr(m, m->leaf_head_scale), leaf_ptr(m, m->leaf_head_bias), m->pooled_f.p, batch, T, D, c.pool, VITB200_DT_F32, m->eps))) return rc;
  mark(m, st, VITB200_CAT_GEMM_HEAD);
  return launch_gemm_f32(st, m->pooled_f.p, leaf_ptr(m, m->head.leaf_kernel), leaf_ptr(m, m->head.leaf_bias), logits, batch, c.num_classes, D, VITB200_EPI_BIAS_F32, nullptr, 0);
}

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace vb_api
using namespace vb_api;

// =============================================================== C ABI ======
extern "C" {

int vitb200_abi_version(void) { return VITB200_ABI_VERSION; }
const char* vitb200_last_error(void) { return last_error_ref().c_str(); }
int64_t vitb200_launch_count(void) { return launch_count(); }

int vitb200_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(VITB200_ERR_NO_DEVICE, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)); }
  int ok = 0;
  for (int d = 0; d < n; ++d) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++ok;
  }
  return ok;
}

int vitb200_create(const vitb200_config* cfg, int device, vitb200_model** out) {
  if (!cfg || !out) return fail(VITB200_ERR_INVALID, "create: null argument");
  *out = nullptr;
  const vitb200_config& c = *cfg;
  if (c.image_h <= 0 || c.image_w <= 0 || c.patch_h <= 0 || c.patch_w <= 0 || c.channels <= 0 ||
      c.num_classes <= 0 || c.dim <= 0 || c.depth < 0 || c.heads <= 0 || c.mlp_dim <= 0 || c.max_batch <= 0)
    return fail(VITB200_ERR_INVALID, "create: non-positive field in config");
  if (c.image_h % c.patch_h != 0 || c.image_w % c.patch_w != 0)      // vit.py:133-134
    return fail(VITB200_ERR_INVALID, "create: image dimensions must be divisible by the patch size");
  if (c.pool != VITB200_POOL_CLS && c.pool != VITB200_POOL_MEAN)     // vit.py:137
    return fail(VITB200_ERR_INVALID, "create: pool must be cls or mean");
  if (c.precision != VITB200_PREC_BF16 && c.precision != VITB200_PREC_FP32 && c.precision != VITB200_PREC_FP16 &&
      c.precision != VITB200_PREC_FP8)
    return fail(VITB200_ERR_INVALID, "create: unknown precision");
  if (!(c.dropout >= 0.f && c.dropout < 1.f) || !(c.emb_dropout >= 0.f && c.emb_dropout < 1.f))
    return fail(VITB200_ERR_INVALID, "create: dropout rates must be in [0, 1)");
  if (c.precision == VITB200_PREC_FP8 && (c.dropout > 0.f || c.emb_dropout > 0.f))
    return fail(VITB200_ERR_UNSUPPORTED, "create: the fp8 precision is an inference forward: dropout rates must be 0");
  if (c.precision == VITB200_PREC_FP8 && (c.dim % 16 != 0 || c.mlp_dim % 16 != 0))
    return fail(VITB200_ERR_UNSUPPORTED, "create: the fp8 precision needs dim and mlp_dim to be multiples of 16 (E4M3 rows "
                                         "of a 16-byte pitch)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return fail(VITB200_ERR_NO_DEVICE, "create: no CUDA device visible (this library has no CPU fallback)");
  }
  if (device < 0 || device >= ndev) return fail(VITB200_ERR_INVALID, "create: device index out of range");
  int major = 0;
  VB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(VITB200_ERR_NO_DEVICE, "create: device is not sm_100 (B200); kernels are sm_100a only");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(VITB200_ERR_CUDA, "create: cudaSetDevice failed");

  std::unique_ptr<vitb200_model> m(new vitb200_model());
  m->cfg = c;
  m->device = device;
  m->Np = (c.image_h / c.patch_h) * (c.image_w / c.patch_w);
  m->cls_off = (c.flags & VITB200_FLAG_NO_CLS) ? 0 : 1;
  m->nchw = (c.flags & VITB200_FLAG_NCHW) ? 1 : 0;
  m->eps = c.ln_eps > 0.f ? c.ln_eps : 1e-6f;
  m->T = m->Np + m->cls_off;
  m->K0 = c.patch_h * c.patch_w * c.channels;
  m->tc = c.precision != VITB200_PREC_FP32;
  m->fp8 = c.precision == VITB200_PREC_FP8;
  m->dt = (c.precision == VITB200_PREC_FP16 || m->fp8) ? VITB200_DT_F16 : VITB200_DT_BF16;
  m->K0pad = m->tc ? int(round_up(m->K0, GEMM_BK)) : m->K0 + (m->K0 & 1);
  m->inner = DIM_HEAD * c.heads;
  m->project_out = !(c.heads == 1 && DIM_HEAD == c.dim);             // vit.py:65
  m->head_tc = m->tc && (c.num_classes % 8 == 0);
  {  // Fused im2col patch embedding (patch_tc.cu): NHWC images whose patch rows are whole 16-byte-aligned TMA runs (every
     // /16 config).  OPT-IN (VITB200_IM2COL=1): measured on B200 at ViT-B/16 batch 256 it takes 0.29 ms against 0.06 +
     // 0.15 ms for patchify + the TOKENS GEMM -- an im2col-mode load is one 192-byte request per (patch, patch row), 2.4 M
     // requests per n-tile pass, and the TMA unit is the bottleneck (profiles/r02_patch_embed.md).
    const char* e = getenv("VITB200_IM2COL");
    m->im2col = m->tc && !m->nchw && c.emb_dropout == 0.f && c.patch_h <= 16 &&
                patch_im2col_supported(c.patch_w, c.channels, c.dim) && (e && e[0] == '1');
  }
  {  // LayerNorm fold: on by default for the dropout-free inference forward; VITB200_LN_FOLD=0 keeps the LayerNorm kernel (A/B)
    const char* e = getenv("VITB200_LN_FOLD");
    // fp8 keeps the LayerNorm kernel: it holds a whole row and emits the bounded, normalised values E4M3 can carry
    m->fold = m->tc && !m->fp8 && m->project_out && c.depth > 0 && c.dropout == 0.f && c.emb_dropout == 0.f && !(e && e[0] == '0');
  }
  if (m->tc && (c.dim % 8 != 0 || c.mlp_dim % 8 != 0))
    return fail(VITB200_ERR_UNSUPPORTED, "create: bf16/fp16 modes need dim and mlp_dim to be multiples of 8");
  if (!m->tc && m->K0pad != m->K0)
    return fail(VITB200_ERR_UNSUPPORTED, "create: fp32 mode needs an even patch feature count");
  build_registry(m.get());
  m->leaf_flags.assign(m->leaves.size(), VITB200_LEAF_TRAINABLE | VITB200_LEAF_DECAY);
  int rc = alloc_workspace(m.get());
  if (rc) return rc;
  *out = m.release();
  return 0;
}

int vitb200_destroy(vitb200_model* m) {
  if (!m) return 0;
  DeviceGuard guard(m->device);
  delete m;
  return 0;
}

int vitb200_num_params(const vitb200_model* m) {
  if (!m) return fail(VITB200_ERR_INVALID, "num_params: null model");
  return int(m->leaves.size());
}

int vitb200_param_info(const vitb200_model* m, int index, const char** path, int64_t shape[4]) {
  if (!m || index < 0 || index >= int(m->leaves.size())) return fail(VITB200_ERR_INVALID, "param_info: bad index");
  const Leaf& l = m->leaves[index];
  if (path) *path = l.path.c_str();
  if (shape) for (size_t i = 0; i < 4; ++i) shape[i] = i < l.shape.size() ? l.shape[i] : 0;
  return int(l.shape.size());
}

int vitb200_set_param(vitb200_model* m, const char* path, const float* host_data, const int64_t* shape, int ndim) {
  if (!m || !path || !host_data || !shape) return fail(VITB200_ERR_INVALID, "set_param: null argument");
  auto it = m->index.find(path);
  if (it == m->index.end()) return fail(VITB200_ERR_INVALID, std::string("set_param: unknown parameter path '") + path + "'");
  Leaf& l = m->leaves[it->second];
  bool same = ndim == int(l.shape.size());
  for (int i = 0; same && i < ndim; ++i) same = shape[i] == l.shape[i];
  if (!same) {
    std::string want, got;
    for (auto s : l.shape) want += std::to_string(s) + ",";
    for (int i = 0; i < ndim; ++i) got += std::to_string(shape[i]) + ",";
    return fail(VITB200_ERR_INVALID, std::string("set_param: shape mismatch for '") + path + "': expected (" + want + ") got (" + got + ")");
  }
  DeviceGuard guard(m->device);
  if (!l.dev) VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&l.dev), size_t(l.numel()) * sizeof(float)));
  VB_CUDA(cudaMemcpy(l.dev, host_data, size_t(l.numel()) * sizeof(float), cudaMemcpyHostToDevice));
  l.set = true;
  m->finalized = false;
  return 0;
}

int vitb200_finalize_params(vitb200_model* m, void* stream) {
  if (!m) return fail(VITB200_ERR_INVALID, "finalize_params: null model");
  for (const auto& l : m->leaves)
    if (!l.set) return fail(VITB200_ERR_PARAM_MISSING, "finalize_params: parameter '" + l.path + "' was never set");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (m->tc) {
    int rc;
    if ((rc = pack_dense(m, m->patch, st))) return rc;
    for (auto& L : m->layers) {
      if (m->fp8) {   // E4M3 codes + column scales for to_qkv and the FeedForward; no 16-bit packs of those three
        if ((rc = quant_dense(m, L.qkv, st)) || (rc = quant_dense(m, L.ff1, st)) || (rc = quant_dense(m, L.ff2, st))) return rc;
        if ((rc = pack_dense(m, L.out, st))) return rc;
        continue;
      }
      if ((rc = pack_dense(m, L.qkv, st))) return rc;
      if ((rc = pack_dense(m, L.out, st))) return rc;
      if ((rc = pack_dense(m, L.ff1, st))) return rc;
      if ((rc = pack_dense(m, L.ff2, st))) return rc;
    }
    if (m->head_tc && (rc = pack_dense(m, m->head, st))) return rc;
    if (m->im2col) {
      const auto& c = m->cfg;
      const int run = c.patch_w * c.channels, kp = c.patch_h * 64;
      if (!m->patch_wt_i2c) VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&m->patch_wt_i2c), size_t(c.dim) * kp * sizeof(uint16_t)));
      if ((rc = launch_pack_weight_im2col(st, m->leaves[m->patch.leaf_kernel].dev, m->patch_wt_i2c, c.dim, c.patch_h, run, m->dt))) return rc;
      if ((rc = make_tmap_2d(&m->patch_tm_i2c, m->patch_wt_i2c, c.dim, kp, kp, GEMM_BN, m->dt))) return rc;
    }
    if (m->fold) {
      DevBuf<float> scratch;
      if ((rc = scratch.alloc(fold_scratch_floats(m)))) return rc;
      for (auto& L : m->layers) {
        if ((rc = fold_dense(m, L.qkv, L.ln1_scale, L.ln1_bias, scratch.p, st))) return rc;
        if ((rc = fold_dense(m, L.ff1, L.ln2_scale, L.ln2_bias, scratch.p, st))) return rc;
      }
      VB_CUDA(cudaStreamSynchronize(st));      // scratch is freed on return
    }
  }
  VB_CUDA(cudaStreamSynchronize(st));
  // graphs captured before a reload hold the old tensor maps and leaf pointers
  for (auto& g : m->graphs)
    for (auto& e : g.second.entries)
      if (e.exec) cudaGraphExecDestroy(e.exec);
  m->graphs.clear();
  m->finalized = true;
  return 0;
}

// ---- graph replay of the forward (launch-bound sizes) -------------------------------------------
// At batch 1 the 88 kernels of a ViT-B/16 forward take less time on the GPU than their launches do
// on the CPU; replaying them as one instantiated graph (programmatic-dependent-launch edges are kept
// by stream capture) removes the per-launch cost.  Large batches gain nothing (the GPU is the
// bottleneck) and are launched directly.  VITB200_GRAPH=0 turns graphs off, =1 forces them for every size.
namespace {
constexpr int64_t kGraphMaxRows = 8192;      // token rows; above this a forward is GPU-bound
constexpr size_t kGraphsPerBatch = 4;        // (images, logits) pairs kept per batch size
constexpr int kGraphMaxCaptures = 16;        // per batch size; beyond this the caller's buffers do not repeat

int graph_mode() {
  static int mode = -1;
  if (mode < 0) {
    const char* e = getenv("VITB200_GRAPH");
    mode = e ? (atoi(e) == 0 ? 0 : 2) : 1;   // 0 off, 1 auto (small sizes), 2 always
  }
  return mode;
}

bool graph_eligible(vitb200_model* m, cudaStream_t st, int batch) {
  const int mode = graph_mode();
  if (mode == 0 || m->prof) return false;
  if (m->cfg.dropout > 0.f || m->cfg.emb_dropout > 0.f) return false;   // the key is a kernel argument
  if (mode == 1 && int64_t(batch) * m->T > kGraphMaxRows) return false;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
  if (cs != cudaStreamCaptureStatusNone) return false;                  // the caller is building its own graph
  auto it = m->graphs.find(batch);
  return it == m->graphs.end() || it->second.captures <= kGraphMaxCaptures;
}

int forward_graph(vitb200_model* m, cudaStream_t st, const float* images, int batch, float* logits) {
  vitb200_model::GraphSlot& slot = m->graphs[batch];
  vitb200_model::FwdGraph* hit = nullptr;
  for (auto& e : slot.entries)
    if (e.images == images && e.logits == logits) hit = &e;
  if (!hit) {
    if (++slot.captures > kGraphMaxCaptures) return forward_tc(m, st, images, batch, logits);
    if (!m->capture_stream) VB_CUDA(cudaStreamCreateWithFlags(&m->capture_stream, cudaStreamNonBlocking));
    // captured on a private stream (the caller's may be the legacy default stream, which cannot capture)
    VB_CUDA(cudaStreamBeginCapture(m->capture_stream, cudaStreamCaptureModeThreadLocal));
    const int rc = forward_tc(m, m->capture_stream, images, batch, logits);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(m->capture_stream, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (ce != cudaSuccess) return cuda_fail(ce, "forward: cudaStreamEndCapture");
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) return cuda_fail(ie, "forward: cudaGraphInstantiate");
    if (slot.entries.size() >= kGraphsPerBatch) {       // evict the least recently used pair
      size_t lru = 0;
      for (size_t i = 1; i < slot.entries.size(); ++i)
        if (slot.entries[i].last_use < slot.entries[lru].last_use) lru = i;
      cudaGraphExecDestroy(slot.entries[lru].exec);
      slot.entries.erase(slot.entries.begin() + lru);
    }
    slot.entries.push_back({images, logits, exec, 0});
    hit = &slot.entries.back();
  }
  hit->last_use = ++m->graph_clock;
  VB_CUDA(cudaGraphLaunch(hit->exec, st));
  return 0;
}
}  // namespace

int vitb200_set_dropout_key(vitb200_model* m, uint64_t key) {
  if (!m) return fail(VITB200_ERR_INVALID, "set_dropout_key: null model");
  m->dropout_key = key;
  return 0;
}

int vitb200_forward(vitb200_model* m, void* stream, const float* images_dev, int batch, float* logits_dev) {
  if (!m || !images_dev || !logits_dev) return fail(VITB200_ERR_INVALID, "forward: null argument");
  if (!m->finalized) return fail(VITB200_ERR_PARAM_MISSING, "forward: call finalize_params first");
  if (batch <= 0 || batch > m->cfg.max_batch) return fail(VITB200_ERR_INVALID, "forward: batch must be in [1, max_batch]");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // an inference forward re-uses the patch matrix a pending backward would read: that backward is now refused
  if (m->train && m->train->fwd_batch != 0) { m->train->fwd_batch = 0; m->train->stale = true; }
  m->tokens_partial = cls_tail(m, nullptr);
  if (!m->tc) return forward_f32(m, st, images_dev, batch, logits_dev);
  if (graph_eligible(m, st, batch)) return forward_graph(m, st, images_dev, batch, logits_dev);
  return forward_tc(m, st, images_dev, batch, logits_dev);
}

int vitb200_forward_attn(vitb200_model* m, void* stream, const float* images_dev, int batch, float* logits_dev,
                         const int* layers, int n_layers, float* maps_dev) {
  if (!m || !images_dev || !logits_dev || !layers || !maps_dev) return fail(VITB200_ERR_INVALID, "forward_attn: null argument");
  if (!m->finalized) return fail(VITB200_ERR_PARAM_MISSING, "forward_attn: call finalize_params first");
  if (batch <= 0 || batch > m->cfg.max_batch) return fail(VITB200_ERR_INVALID, "forward_attn: batch must be in [1, max_batch]");
  const int depth = m->cfg.depth;
  if (n_layers <= 0 || n_layers > depth) return fail(VITB200_ERR_INVALID, "forward_attn: n_layers must be in [1, depth]");
  AttnRecord rec;
  rec.slot.assign(size_t(depth), -1);
  rec.n = n_layers;
  rec.maps = maps_dev;
  for (int i = 0; i < n_layers; ++i) {
    const int l = layers[i];
    if (l < 0 || l >= depth) return fail(VITB200_ERR_INVALID, "forward_attn: layer index outside [0, depth)");
    if (rec.slot[size_t(l)] >= 0) return fail(VITB200_ERR_INVALID, "forward_attn: a layer is listed twice");
    rec.slot[size_t(l)] = i;
  }
  if (!m->tc) return fail(VITB200_ERR_UNSUPPORTED, "forward_attn: the fp32 validation path does not record attention maps");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (m->attn_lse.n == 0) {
    int rc;
    if ((rc = m->attn_lse.alloc(size_t(m->cfg.max_batch) * m->cfg.heads * m->T))) return rc;
  }
  // the same workspace as vitb200_forward: a pending backward is refused afterwards
  if (m->train && m->train->fwd_batch != 0) { m->train->fwd_batch = 0; m->train->stale = true; }
  m->tokens_partial = cls_tail(m, &rec);
  // launched directly: a recording forward neither replays nor captures the forward graphs
  return forward_tc(m, st, images_dev, batch, logits_dev, &rec);
}

int vitb200_forward_host(vitb200_model* m, void* stream, const float* images_host, int batch, float* logits_host) {
  if (!m || !images_host || !logits_host) return fail(VITB200_ERR_INVALID, "forward_host: null argument");
  if (batch <= 0 || batch > m->cfg.max_batch) return fail(VITB200_ERR_INVALID, "forward_host: batch must be in [1, max_batch]");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto& c = m->cfg;
  const size_t img_elems = size_t(c.max_batch) * c.image_h * c.image_w * c.channels;
  int rc;
  if (m->img_stage.n < img_elems && (rc = m->img_stage.alloc(img_elems))) return rc;
  if (m->logit_stage.n < size_t(c.max_batch) * c.num_classes && (rc = m->logit_stage.alloc(size_t(c.max_batch) * c.num_classes))) return rc;
  const size_t in_bytes = size_t(batch) * c.image_h * c.image_w * c.channels * sizeof(float);
  const size_t out_bytes = size_t(batch) * c.num_classes * sizeof(float);
  VB_CUDA(cudaMemcpyAsync(m->img_stage.p, images_host, in_bytes, cudaMemcpyHostToDevice, st));
  if ((rc = vitb200_forward(m, stream, m->img_stage.p, batch, m->logit_stage.p))) return rc;
  VB_CUDA(cudaMemcpyAsync(logits_host, m->logit_stage.p, out_bytes, cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int vitb200_submit_host(vitb200_model* m, void* stream, const float* images_host, int batch, float* logits_host) {
  if (!m || !images_host || !logits_host) return fail(VITB200_ERR_INVALID, "submit_host: null argument");
  if (batch <= 0 || batch > m->cfg.max_batch) return fail(VITB200_ERR_INVALID, "submit_host: batch must be in [1, max_batch]");
  if (m->jobs_submitted - m->jobs_waited >= 2) return fail(VITB200_ERR_INVALID, "submit_host: two jobs already in flight, call wait_host first");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto& c = m->cfg;
  int rc;
  if (!m->h2d_stream) {
    VB_CUDA(cudaStreamCreateWithFlags(&m->h2d_stream, cudaStreamNonBlocking));
    VB_CUDA(cudaStreamCreateWithFlags(&m->d2h_stream, cudaStreamNonBlocking));
  }
  vitb200_model::HostJob& j = m->job[m->jobs_submitted & 1];
  const size_t img_elems = size_t(c.max_batch) * c.image_h * c.image_w * c.channels;
  if (j.img.n < img_elems && (rc = j.img.alloc(img_elems))) return rc;
  if (j.logit.n < size_t(c.max_batch) * c.num_classes && (rc = j.logit.alloc(size_t(c.max_batch) * c.num_classes))) return rc;
  if (!j.h2d_done) {
    VB_CUDA(cudaEventCreateWithFlags(&j.h2d_done, cudaEventDisableTiming));
    VB_CUDA(cudaEventCreateWithFlags(&j.fwd_done, cudaEventDisableTiming));
    VB_CUDA(cudaEventCreateWithFlags(&j.d2h_done, cudaEventDisableTiming));
  }
  const size_t in_bytes = size_t(batch) * c.image_h * c.image_w * c.channels * sizeof(float);
  const size_t out_bytes = size_t(batch) * c.num_classes * sizeof(float);
  // H2D on its own stream: the slot's previous forward (two jobs ago) has read its images
  if (j.used) VB_CUDA(cudaStreamWaitEvent(m->h2d_stream, j.fwd_done, 0));
  VB_CUDA(cudaMemcpyAsync(j.img.p, images_host, in_bytes, cudaMemcpyHostToDevice, m->h2d_stream));
  VB_CUDA(cudaEventRecord(j.h2d_done, m->h2d_stream));
  // forward on the caller's stream: images have landed, the slot's previous logits have left
  VB_CUDA(cudaStreamWaitEvent(st, j.h2d_done, 0));
  if (j.used) VB_CUDA(cudaStreamWaitEvent(st, j.d2h_done, 0));
  if ((rc = vitb200_forward(m, stream, j.img.p, batch, j.logit.p))) return rc;
  VB_CUDA(cudaEventRecord(j.fwd_done, st));
  // D2H on its own stream
  VB_CUDA(cudaStreamWaitEvent(m->d2h_stream, j.fwd_done, 0));
  VB_CUDA(cudaMemcpyAsync(logits_host, j.logit.p, out_bytes, cudaMemcpyDeviceToHost, m->d2h_stream));
  VB_CUDA(cudaEventRecord(j.d2h_done, m->d2h_stream));
  j.used = true;
  j.pending = true;
  ++m->jobs_submitted;
  return 0;
}

int vitb200_wait_host(vitb200_model* m) {
  if (!m) return fail(VITB200_ERR_INVALID, "wait_host: null model");
  if (m->jobs_waited >= m->jobs_submitted) return fail(VITB200_ERR_INVALID, "wait_host: nothing in flight");
  DeviceGuard guard(m->device);
  vitb200_model::HostJob& j = m->job[m->jobs_waited & 1];
  VB_CUDA(cudaEventSynchronize(j.d2h_done));
  j.pending = false;
  ++m->jobs_waited;
  return 0;
}

int vitb200_profile_forward(vitb200_model* m, void* stream, const float* images_dev, int batch, float* logits_dev,
                            float* ms_by_category, int* launches_by_category) {
  if (!m || !ms_by_category || !launches_by_category) return fail(VITB200_ERR_INVALID, "profile_forward: null argument");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<std::pair<int, cudaEvent_t>> marks;
  marks.reserve(512);
  m->prof = &marks;
  int rc = vitb200_forward(m, stream, images_dev, batch, logits_dev);
  mark(m, st, -1);
  m->prof = nullptr;
  cudaError_t e = cudaStreamSynchronize(st);
  for (int c = 0; c < VITB200_NUM_CATEGORIES; ++c) { ms_by_category[c] = 0.f; launches_by_category[c] = 0; }
  if (rc == 0 && e == cudaSuccess) {
    for (size_t i = 0; i + 1 < marks.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, marks[i].second, marks[i + 1].second);
      const int c = marks[i].first;
      if (c >= 0 && c < VITB200_NUM_CATEGORIES) { ms_by_category[c] += ms; launches_by_category[c] += 1; }
    }
  }
  for (auto& mk : marks) cudaEventDestroy(mk.second);
  if (rc) return rc;
  if (e != cudaSuccess) return cuda_fail(e, "profile_forward: cudaStreamSynchronize");
  return 0;
}

int vitb200_debug_tokens(vitb200_model* m, void* stream, float* tokens_host, int batch) {
  if (!m || !tokens_host) return fail(VITB200_ERR_INVALID, "debug_tokens: null argument");
  if (batch <= 0 || batch > m->cfg.max_batch) return fail(VITB200_ERR_INVALID, "debug_tokens: bad batch");
  if (m->tokens_partial)
    return fail(VITB200_ERR_UNSUPPORTED, "debug_tokens: the last forward ran the class-token tail (pool = 'cls'): its last "
                                         "block computed only the class-token rows, the other rows are stale.  A forward that "
                                         "records the last layer's attention weights (vitb200_forward_attn) runs it in full");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  VB_CUDA(cudaMemcpyAsync(tokens_host, m->x.p, size_t(batch) * m->T * m->cfg.dim * sizeof(float), cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ---- training: a forward that keeps its activations, and the backward pass (SURVEY.md section 8f-4) ----
// Nothing in the reference trains, so there is no reference API to mirror; the C entry points are
// the two halves of jax.vjp(lambda p: ViT.apply(p, img), params): train_forward returns the logits,
// backward takes their cotangent and fills one fp32 gradient per parameter leaf.
namespace {

inline float* grad_ptr(vitb200_model* m, int leaf) { return leaf >= 0 ? m->train->grads.p + m->train->grad_off[leaf] : nullptr; }

// C[c_rows <= M, N] = epilogue(A[M, K] x Wt[N, ldw]^T) with tensor maps encoded per call (host side, ~1 us each)
int gemm16(vitb200_model* m, cudaStream_t st, const void* A, int M, int K, const void* Wt, int ldw, int N, void* C,
           int c_rows, int epi, const float* bias, const float* aux = nullptr, int tpi = 0, const float* cls = nullptr,
           const Dropout& drop = Dropout()) {
  CUtensorMap ta, tb, tc;
  int rc;
  const int cg = gemm_tc_tile_mode(M, N);
  const bool out16 = epi == VITB200_EPI_STORE_16 || epi == VITB200_EPI_BIAS_GELU_16 || epi == VITB200_EPI_BIAS_16 ||
                     epi == VITB200_EPI_BIAS_PRE_GELU_16;
  if ((rc = make_tmap_2d(&ta, A, M, K, K, GEMM_BM, m->dt))) return rc;
  if ((rc = make_tmap_2d(&tb, Wt, N, ldw, ldw, cg == 64 ? 64 : GEMM_BN / cg, m->dt))) return rc;
  if ((rc = make_tmap_2d(&tc, C, c_rows, N, N, GEMM_BM, out16 ? m->dt : VITB200_DT_F32))) return rc;
  return launch_gemm_tc(st, ta, tb, &tc, bias, C, M, N, K, epi, aux, tpi, m->dt, cg, drop, m->cls_off, cls);
}

// dW[Dx (first c_rows rows), Dy] += X[R, Dx]^T dY[R, Dy]: the GEMM reads both row-major activations as
// MN-major operands (K = the row index), split-K so that the few output tiles of a weight gradient
// (9 for 768 x 768) become about two waves of work; the partial sums meet in the TMA reduce-add.
// VITB200_WGRAD_TRANSPOSE=1 keeps the first implementation (explicit transposed copies + the K-major GEMM).
int wgrad(vitb200_model* m, cudaStream_t st, const void* X, int Dx, const void* dY, int Dy, int R, float* dW, int c_rows) {
  auto& ts = *m->train;
  const int cg = gemm_tc_tile_mode(Dx, Dy) == 4 ? 2 : gemm_tc_tile_mode(Dx, Dy);
  const int tm = cg == 2 ? 2 * GEMM_BM : GEMM_BM, tn = cg == 64 ? 64 : GEMM_BN, units = cg == 2 ? sm_count() / 2 : sm_count();
  const int mn_tiles = ceil_div(Dx, tm) * ceil_div(Dy, tn);
  const int splits = std::max(1, 2 * units / mn_tiles);
  static const bool via_transpose = [] { const char* e = getenv("VITB200_WGRAD_TRANSPOSE"); return e && e[0] == '1'; }();
  int rc;
  if (via_transpose) {
    const int Rpad = int(round_up(R, 64));
    if ((rc = launch_transpose16(st, X, ts.tA.p, R, Dx, Rpad))) return rc;
    if ((rc = launch_transpose16(st, dY, ts.tB.p, R, Dy, Rpad))) return rc;
    return gemm16(m, st, ts.tA.p, Dx, Rpad, ts.tB.p, Rpad, Dy, dW, c_rows, VITB200_EPI_BIAS_RESID_F32, ts.zeros.p, nullptr, splits);
  }
  CUtensorMap tx, ty, tc;
  if ((rc = make_tmap_2d(&tx, X, R, Dx, Dx, 64, m->dt))) return rc;
  if ((rc = make_tmap_2d(&ty, dY, R, Dy, Dy, 64, m->dt))) return rc;
  if ((rc = make_tmap_2d(&tc, dW, c_rows, Dy, Dy, GEMM_BM, VITB200_DT_F32))) return rc;
  return launch_gemm_tc_wgrad(st, tx, ty, tc, ts.zeros.p, dW, Dx, Dy, R, splits, m->dt, cg);
}

int train_supported(const vitb200_model* m) {
  const auto& c = m->cfg;
  if (!m->tc) return fail(VITB200_ERR_UNSUPPORTED, "train: the backward pass is built for the bf16/fp16 modes only");
  if (m->fp8) return fail(VITB200_ERR_UNSUPPORTED, "train: the fp8 precision is inference only (train in fp16 or bf16)");
  if (!m->project_out) return fail(VITB200_ERR_UNSUPPORTED, "train: heads == 1 with dim == 64 (identity to_out) is not built");
  if (c.dim > 1280) return fail(VITB200_ERR_UNSUPPORTED, "train: dim > 1280 is not built for the backward pass");
  if (c.depth < 1) return fail(VITB200_ERR_UNSUPPORTED, "train: the backward pass needs at least one transformer layer");
  return 0;
}

int ensure_train(vitb200_model* m, cudaStream_t st) {
  if (m->train) return 0;
  const auto& c = m->cfg;
  std::unique_ptr<vitb200_model::TrainState> ts(new vitb200_model::TrainState());
  const size_t B = size_t(c.max_batch), R = B * m->T, Rpad = size_t(round_up(int64_t(R), 64));
  const size_t D = size_t(c.dim), I = size_t(m->inner), H = size_t(c.mlp_dim);
  int rc;
  ts->xs.resize(2 * size_t(c.depth) + 1);
  for (auto& x : ts->xs) if ((rc = x.alloc(R * D))) return rc;
  ts->layers.resize(size_t(c.depth));
  ts->rows_cap = int(round_up(int64_t(R), 2 * GEMM_BM));
  for (auto& L : ts->layers) {
    if ((rc = L.xn1.alloc(R * D)) || (rc = L.qkv.alloc(R * 3 * I)) || (rc = L.o.alloc(R * I)) ||
        (rc = L.xn2.alloc(R * D)) || (rc = L.pre.alloc(2 * size_t(ts->rows_cap) * H))) return rc;
    if ((rc = L.lse.alloc(B * size_t(c.heads) * m->T))) return rc;
    L.hid = L.pre.p + size_t(ts->rows_cap) * H;
  }
  if ((rc = ts->dx.alloc(R * D)) || (rc = ts->pooled_ln.alloc(B * D)) || (rc = ts->dpl.alloc(B * D))) return rc;
  if ((rc = ts->dy16.alloc(R * D)) || (rc = ts->dhid16.alloc(R * H)) || (rc = ts->dxn16.alloc(R * D)) ||
      (rc = ts->do16.alloc(R * I)) || (rc = ts->dqkv16.alloc(R * 3 * I))) return rc;
  if ((rc = ts->attn_ws.alloc(attention_bwd_workspace_floats(c.max_batch, m->T, c.heads)))) return rc;   // D (+ fp32 dQ beyond 208 tokens)
  const size_t dx_max = std::max(std::max(H, D), std::max(I, size_t(m->K0pad))), dy_max = std::max(std::max(H, D), 3 * I);
  if ((rc = ts->tA.alloc(dx_max * Rpad)) || (rc = ts->tB.alloc(dy_max * Rpad))) return rc;
  const size_t nz = std::max(std::max(dx_max, dy_max), size_t(c.num_classes));
  if ((rc = ts->zeros.alloc(nz))) return rc;
  VB_CUDA(cudaMemsetAsync(ts->zeros.p, 0, nz * sizeof(float), st));
  size_t total = 0;
  for (const auto& l : m->leaves) {
    ts->grad_off.push_back(total);
    total += size_t(round_up(l.numel(), 64));        // 256-byte aligned leaves (TMA reduce-add targets)
  }
  if ((rc = ts->grads.alloc(total))) return rc;
  VB_CUDA(cudaMemsetAsync(ts->grads.p, 0, total * sizeof(float), st));
  // Flax-layout 16-bit weight copies for the dgrad GEMMs
  auto make_wf = [&](DenseW& d) -> int {
    if (d.leaf_kernel < 0) return 0;
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.wf), size_t(d.K) * d.N * sizeof(uint16_t)));
    return launch_cast16(st, m->leaves[d.leaf_kernel].dev, d.wf, int64_t(d.K) * d.N, m->dt);
  };
  for (auto& L : m->layers)
    if ((rc = make_wf(L.qkv)) || (rc = make_wf(L.out)) || (rc = make_wf(L.ff1)) || (rc = make_wf(L.ff2))) return rc;
  {  // the patch Dense's copy (image gradients: dpatches = dY W^T) has K0pad rows, the ones past K0 zero, so that its
     // output rows have the K0pad pitch of the patch matrix (an fp32 pitch of K0 = 147 floats is no legal TMA stride)
    DenseW& d = m->patch;
    const size_t n = size_t(m->K0pad) * d.N;
    VB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d.wf), n * sizeof(uint16_t)));
    VB_CUDA(cudaMemsetAsync(d.wf, 0, n * sizeof(uint16_t), st));
    if ((rc = launch_cast16(st, m->leaves[d.leaf_kernel].dev, d.wf, int64_t(d.K) * d.N, m->dt))) return rc;
  }
  m->train = std::move(ts);
  return 0;
}

}  // namespace

int vitb200_train_forward(vitb200_model* m, void* stream, const float* images, int batch, float* logits) {
  if (!m || !images || !logits) return fail(VITB200_ERR_INVALID, "train_forward: null argument");
  if (!m->finalized) return fail(VITB200_ERR_PARAM_MISSING, "train_forward: call finalize_params first");
  if (batch <= 0 || batch > m->cfg.max_batch) return fail(VITB200_ERR_INVALID, "train_forward: batch must be in [1, max_batch]");
  int rc;
  if ((rc = train_supported(m))) return rc;
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = ensure_train(m, st))) return rc;
  auto& ts = *m->train;
  ts.fwd_batch = 0;
  ts.stale = false;
  const auto& c = m->cfg;
  const int D = c.dim, I = m->inner, T = m->T, H = c.mlp_dim, R = batch * T;
  if ((rc = launch_patchify(st, images, m->patches_h.p, batch, c.image_h, c.image_w, c.channels, c.patch_h, c.patch_w,
                            m->K0pad, m->dt, m->nchw, m->cls_off))) return rc;
  if ((rc = gemm16(m, st, m->patches_h.p, R, m->K0pad, m->patch.wt, m->patch.Kpad, D, ts.xs[0].p, R, VITB200_EPI_TOKENS_F32,
                   leaf_ptr(m, m->patch.leaf_bias), leaf_ptr(m, m->leaf_pos), T, leaf_ptr(m, m->leaf_cls),
                   m->drop(c.emb_dropout, 0)))) return rc;
  for (int l = 0; l < c.depth; ++l) {
    Layer& L = m->layers[l];
    auto& S = ts.layers[l];
    float* x0 = ts.xs[2 * l].p;
    float* x1 = ts.xs[2 * l + 1].p;
    float* x2 = ts.xs[2 * l + 2].p;
    // x1 = x0 + to_out(attention(to_qkv(LN1(x0))));  x0 stays behind as the saved LayerNorm input
    if ((rc = launch_layernorm(st, x0, leaf_ptr(m, L.ln1_scale), leaf_ptr(m, L.ln1_bias), S.xn1.p, R, D, m->dt, m->eps, x1))) return rc;
    if ((rc = gemm16(m, st, S.xn1.p, R, D, L.qkv.wt, L.qkv.Kpad, 3 * I, S.qkv.p, R, VITB200_EPI_STORE_16, nullptr))) return rc;
    if ((rc = launch_attention_tc(st, S.qkv.p, S.o.p, batch, T, c.heads, m->dt, S.lse.p))) return rc;
    if ((rc = gemm16(m, st, S.o.p, R, I, L.out.wt, L.out.Kpad, D, x1, R, VITB200_EPI_BIAS_RESID_F32, leaf_ptr(m, L.out.leaf_bias),
                     nullptr, 0, nullptr, m->drop(c.dropout, 1 + 3 * l)))) return rc;
    // x2 = x1 + ff2(gelu(ff1(LN2(x1)))), the pre-activation kept for gelu'
    if ((rc = launch_layernorm(st, x1, leaf_ptr(m, L.ln2_scale), leaf_ptr(m, L.ln2_bias), S.xn2.p, R, D, m->dt, m->eps, x2))) return rc;
    static const bool dual = [] { const char* e = getenv("VITB200_TRAIN_DUAL"); return !(e && e[0] == '0'); }();
    if (dual) {   // one GEMM writes the pre-activation and, rows_cap rows further down the same buffer, its GELU
      if ((rc = gemm16(m, st, S.xn2.p, R, D, L.ff1.wt, L.ff1.Kpad, H, S.pre.p, 2 * ts.rows_cap, VITB200_EPI_BIAS_PRE_GELU_16,
                       leaf_ptr(m, L.ff1.leaf_bias), nullptr, ts.rows_cap, nullptr, m->drop(c.dropout, 2 + 3 * l)))) return rc;
    } else {
      if ((rc = gemm16(m, st, S.xn2.p, R, D, L.ff1.wt, L.ff1.Kpad, H, S.pre.p, R, VITB200_EPI_BIAS_16, leaf_ptr(m, L.ff1.leaf_bias)))) return rc;
      if ((rc = launch_gelu_fwd(st, S.pre.p, S.hid, int64_t(R) * H, m->dt, m->drop(c.dropout, 2 + 3 * l)))) return rc;
    }
    if ((rc = gemm16(m, st, S.hid, R, H, L.ff2.wt, L.ff2.Kpad, D, x2, R, VITB200_EPI_BIAS_RESID_F32, leaf_ptr(m, L.ff2.leaf_bias),
                     nullptr, 0, nullptr, m->drop(c.dropout, 3 + 3 * l)))) return rc;
  }
  const float* xf = ts.xs[2 * size_t(c.depth)].p;
  if ((rc = launch_pool_layernorm(st, xf, leaf_ptr(m, m->leaf_head_scale), leaf_ptr(m, m->leaf_head_bias), ts.pooled_ln.p,
                                  batch, T, D, c.pool, VITB200_DT_F32, m->eps))) return rc;
  if (m->head_tc) {
    if ((rc = launch_pool_layernorm(st, xf, leaf_ptr(m, m->leaf_head_scale), leaf_ptr(m, m->leaf_head_bias), m->pooled_h.p,
                                    batch, T, D, c.pool, m->dt, m->eps))) return rc;
    if ((rc = gemm16(m, st, m->pooled_h.p, batch, D, m->head.wt, m->head.Kpad, c.num_classes, logits, batch, VITB200_EPI_BIAS_F32,
                     leaf_ptr(m, m->head.leaf_bias)))) return rc;
  } else {
    if ((rc = launch_gemm_f32(st, ts.pooled_ln.p, leaf_ptr(m, m->head.leaf_kernel), leaf_ptr(m, m->head.leaf_bias), logits,
                              batch, c.num_classes, D, VITB200_EPI_BIAS_F32, nullptr, 0))) return rc;
  }
  ts.fwd_batch = batch;
  ts.fwd_key = m->dropout_key;
  ts.fwd_version = m->weights_version;
  return 0;
}

namespace {

// One backward schedule for every choice of what to differentiate with respect to.  The chain that carries the
// token-stream cotangent dx from the logits to the images is the same kernels with the same arguments in the same order
// whatever `wrt` is, so image gradients do not depend on whether parameter gradients are computed.  Without
// VITB200_GRAD_PARAMS the weight-gradient GEMMs (4 per layer + the patch kernel's), the head's weight and bias gradients
// and the token-embedding gradients are not launched; the column sums fused into the dx chain's own kernels still land in
// the gradient buffer, which then reads as invalid (vitb200_get_grad & co. refuse).
int backward_impl(vitb200_model* m, cudaStream_t st, const float* dlogits, int batch, int wrt, float* dimages) {
  auto& ts = *m->train;
  const auto& c = m->cfg;
  const int D = c.dim, I = m->inner, T = m->T, H = c.mlp_dim, R = batch * T, dt = m->dt;
  const bool params = (wrt & VITB200_GRAD_PARAMS) != 0, images = (wrt & VITB200_GRAD_IMAGES) != 0;
  int rc;
  if (images && ts.dpatches.n == 0) {   // first image-gradient backward: parameter-only callers never pay for it
    if ((rc = ts.dpatches.alloc(size_t(c.max_batch) * T * m->K0pad))) return rc;
  }
  ts.grads_valid = params;
  ts.grads_fresh = params;
  // the nn.Dropout masks of the forward are pure functions of (key, site, element): replayed, never stored
  const uint64_t cur_key = m->dropout_key;
  m->dropout_key = ts.fwd_key;
  struct KeyRestore { vitb200_model* m; uint64_t k; ~KeyRestore() { m->dropout_key = k; } } restore{m, cur_key};
  VB_CUDA(cudaMemsetAsync(ts.grads.p, 0, ts.grads.n * sizeof(float), st));
  // head: logits = LN(pool(x)) Wh + bh   (vit.py:159-165)
  if ((rc = launch_head_bwd(st, ts.pooled_ln.p, dlogits, leaf_ptr(m, m->head.leaf_kernel),
                            params ? grad_ptr(m, m->head.leaf_kernel) : nullptr, params ? grad_ptr(m, m->head.leaf_bias) : nullptr,
                            ts.dpl.p, batch, D, c.num_classes))) return rc;
  if ((rc = launch_pool_ln_bwd(st, ts.xs[2 * size_t(c.depth)].p, ts.dpl.p, leaf_ptr(m, m->leaf_head_scale), ts.dx.p,
                               grad_ptr(m, m->leaf_head_scale), grad_ptr(m, m->leaf_head_bias), batch, T, D, c.pool, m->eps))) return rc;
  // dy16 = cast(dx) (+ the replayed mask of the Dropout behind FF Dense_1) and its column sums = that bias gradient;
  // for every later stage the LayerNorm adjoint that produces dx emits both itself
  if ((rc = launch_cast16_colsum(st, ts.dx.p, ts.dy16.p, grad_ptr(m, m->layers[c.depth - 1].ff2.leaf_bias), R, D, dt,
                                 m->drop(c.dropout, 3 + 3 * (c.depth - 1))))) return rc;
  for (int l = c.depth - 1; l >= 0; --l) {
    Layer& L = m->layers[l];
    auto& S = ts.layers[l];
    // ---- x2 = x1 + Dense_1(gelu(Dense_0(LN2(x1))))   (vit.py:39,47-53) ----
    if ((rc = gemm16(m, st, ts.dy16.p, R, D, L.ff2.wf, D, H, ts.dhid16.p, R, VITB200_EPI_STORE_16, nullptr))) return rc;
    if (params && (rc = wgrad(m, st, S.hid, H, ts.dy16.p, D, R, grad_ptr(m, L.ff2.leaf_kernel), H))) return rc;
    if ((rc = launch_gelu_bwd_colsum(st, S.pre.p, ts.dhid16.p, ts.dhid16.p, grad_ptr(m, L.ff1.leaf_bias), R, H, dt,
                                     m->drop(c.dropout, 2 + 3 * l)))) return rc;
    if ((rc = gemm16(m, st, ts.dhid16.p, R, H, L.ff1.wf, H, D, ts.dxn16.p, R, VITB200_EPI_STORE_16, nullptr))) return rc;
    if (params && (rc = wgrad(m, st, S.xn2.p, D, ts.dhid16.p, H, R, grad_ptr(m, L.ff1.leaf_kernel), D))) return rc;
    // LayerNorm adjoint; its dx is the cotangent of to_out's output: 16-bit copy + to_out bias gradient ride along
    if ((rc = launch_ln_bwd(st, ts.dxn16.p, ts.xs[2 * l + 1].p, leaf_ptr(m, L.ln2_scale), ts.dx.p, grad_ptr(m, L.ln2_scale),
                            grad_ptr(m, L.ln2_bias), R, D, dt, m->eps, 1, ts.dy16.p, grad_ptr(m, L.out.leaf_bias),
                            m->drop(c.dropout, 1 + 3 * l)))) return rc;
    // ---- x1 = x0 + to_out(attention(to_qkv(LN1(x0))))   (vit.py:39,62-87) ----
    if ((rc = gemm16(m, st, ts.dy16.p, R, D, L.out.wf, D, I, ts.do16.p, R, VITB200_EPI_STORE_16, nullptr))) return rc;
    if (params && (rc = wgrad(m, st, S.o.p, I, ts.dy16.p, D, R, grad_ptr(m, L.out.leaf_kernel), I))) return rc;
    if ((rc = launch_attention_bwd(st, S.qkv.p, S.o.p, ts.do16.p, ts.dqkv16.p, batch, T, c.heads, dt, ts.attn_ws.p, S.lse.p))) return rc;
    if ((rc = gemm16(m, st, ts.dqkv16.p, R, 3 * I, L.qkv.wf, 3 * I, D, ts.dxn16.p, R, VITB200_EPI_STORE_16, nullptr))) return rc;
    if (params && (rc = wgrad(m, st, S.xn1.p, D, ts.dqkv16.p, 3 * I, R, grad_ptr(m, L.qkv.leaf_kernel), D))) return rc;
    // its dx is the cotangent of the previous layer's FF Dense_1 output (layer 0: of the token embedding, handled below)
    if (l > 0) {
      if ((rc = launch_ln_bwd(st, ts.dxn16.p, ts.xs[2 * l].p, leaf_ptr(m, L.ln1_scale), ts.dx.p, grad_ptr(m, L.ln1_scale),
                              grad_ptr(m, L.ln1_bias), R, D, dt, m->eps, 1, ts.dy16.p, grad_ptr(m, m->layers[l - 1].ff2.leaf_bias),
                              m->drop(c.dropout, 3 + 3 * (l - 1))))) return rc;
    } else {
      if ((rc = launch_ln_bwd(st, ts.dxn16.p, ts.xs[0].p, leaf_ptr(m, L.ln1_scale), ts.dx.p, grad_ptr(m, L.ln1_scale),
                              grad_ptr(m, L.ln1_bias), R, D, dt, m->eps, 1))) return rc;
    }
  }
  // ---- tokens = Dropout(concat(cls, patches W + b) + pos)   (vit.py:147-155) ----
  if ((rc = launch_mask_inplace(st, ts.dx.p, int64_t(R) * D, m->drop(c.emb_dropout, 0)))) return rc;
  if (params && (rc = launch_token_grads(st, ts.dx.p, grad_ptr(m, m->leaf_pos), grad_ptr(m, m->leaf_cls),
                                         grad_ptr(m, m->patch.leaf_bias), batch, T, D, m->cls_off))) return rc;
  if ((rc = launch_cast16(st, ts.dx.p, ts.dy16.p, int64_t(R) * D, dt))) return rc;
  // the class-token slot rows of the patch matrix are zero, so their dx rows add nothing to dW
  if (params && (rc = wgrad(m, st, m->patches_h.p, m->K0pad, ts.dy16.p, D, R, grad_ptr(m, m->patch.leaf_kernel), m->K0))) return rc;
  if (images) {
    // ---- patches = patchify(images)   (vit.py:146) ----
    // dpatches [R, K0pad] = dY W^T; the class-token slot rows come out as rows nobody reads, the pad columns as zeros
    if ((rc = gemm16(m, st, ts.dy16.p, R, D, m->patch.wf, D, m->K0pad, ts.dpatches.p, R, VITB200_EPI_BIAS_F32, ts.zeros.p))) return rc;
    if ((rc = launch_unpatchify(st, ts.dpatches.p, dimages, batch, c.image_h, c.image_w, c.channels, c.patch_h, c.patch_w,
                                m->K0pad, m->nchw, m->cls_off))) return rc;
  }
  return 0;
}

int grads_ready(const vitb200_model* m, const char* who) {
  if (!m->train->grads_valid)
    return fail(VITB200_ERR_INVALID, std::string(who) + ": the last backward did not compute parameter gradients "
                                     "(run one with VITB200_GRAD_PARAMS)");
  return 0;
}

}  // namespace

int vitb200_backward_ex(vitb200_model* m, void* stream, const float* dlogits, int batch, int wrt, float* dimages) {
  if (!m || !dlogits) return fail(VITB200_ERR_INVALID, "backward: null argument");
  if (m->fp8) return fail(VITB200_ERR_UNSUPPORTED, "backward: the fp8 precision is inference only (train in fp16 or bf16)");
  if (wrt == 0 || (wrt & ~(VITB200_GRAD_PARAMS | VITB200_GRAD_IMAGES)) != 0)
    return fail(VITB200_ERR_INVALID, "backward: wrt must be a non-zero OR of VITB200_GRAD_PARAMS and VITB200_GRAD_IMAGES");
  if ((wrt & VITB200_GRAD_IMAGES) && !dimages)
    return fail(VITB200_ERR_INVALID, "backward: VITB200_GRAD_IMAGES needs an image-gradient buffer");
  if (m->train && m->train->fwd_batch == 0 && m->train->stale)
    return fail(VITB200_ERR_INVALID, "backward: a forward ran on this handle since train_forward and overwrote its workspace; "
                                     "call train_forward again");
  if (!m->train || m->train->fwd_batch == 0) return fail(VITB200_ERR_INVALID, "backward: call train_forward first");
  if (batch != m->train->fwd_batch) return fail(VITB200_ERR_INVALID, "backward: batch differs from the last train_forward");
  if (m->train->fwd_version != m->weights_version)
    return fail(VITB200_ERR_INVALID, "backward: an optimiser step changed the weights since train_forward; call train_forward again");
  if (!m->finalized) return fail(VITB200_ERR_PARAM_MISSING, "backward: parameters changed since train_forward");
  DeviceGuard guard(m->device);
  return backward_impl(m, static_cast<cudaStream_t>(stream), dlogits, batch, wrt, dimages);
}

int vitb200_backward(vitb200_model* m, void* stream, const float* dlogits, int batch) {
  return vitb200_backward_ex(m, stream, dlogits, batch, VITB200_GRAD_PARAMS, nullptr);
}

int vitb200_get_grad(vitb200_model* m, void* stream, const char* path, float* host_out) {
  if (!m || !path || !host_out) return fail(VITB200_ERR_INVALID, "get_grad: null argument");
  if (!m->train) return fail(VITB200_ERR_INVALID, "get_grad: no backward pass has run");
  if (int rc = grads_ready(m, "get_grad")) return rc;
  auto it = m->index.find(path);
  if (it == m->index.end()) return fail(VITB200_ERR_INVALID, std::string("get_grad: unknown parameter path '") + path + "'");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  VB_CUDA(cudaMemcpyAsync(host_out, grad_ptr(m, it->second), size_t(m->leaves[it->second].numel()) * sizeof(float),
                          cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int vitb200_grads_buffer(vitb200_model* m, float** dev_out, int64_t* count) {
  if (!m || !dev_out || !count) return fail(VITB200_ERR_INVALID, "grads_buffer: null argument");
  if (!m->train) return fail(VITB200_ERR_INVALID, "grads_buffer: no train_forward has run");
  if (int rc = grads_ready(m, "grads_buffer")) return rc;
  *dev_out = m->train->grads.p;
  *count = int64_t(m->train->grads.n);
  return 0;
}

int vitb200_grad_device(vitb200_model* m, const char* path, float** dev_out) {
  if (!m || !path || !dev_out) return fail(VITB200_ERR_INVALID, "grad_device: null argument");
  if (!m->train) return fail(VITB200_ERR_INVALID, "grad_device: no backward pass has run");
  if (int rc = grads_ready(m, "grad_device")) return rc;
  auto it = m->index.find(path);
  if (it == m->index.end()) return fail(VITB200_ERR_INVALID, std::string("grad_device: unknown parameter path '") + path + "'");
  *dev_out = grad_ptr(m, it->second);
  return 0;
}

// ---- on-device training step (optim.cu) ------------------------------------------------------------------------------
namespace {

int check_adamw(const vitb200_adamw& h) {
  auto finite = [](float v) { return std::isfinite(v); };
  if (!finite(h.lr) || h.lr < 0.f) return fail(VITB200_ERR_INVALID, "adamw_step: lr must be finite and >= 0");
  if (!(h.b1 >= 0.f && h.b1 < 1.f) || !(h.b2 >= 0.f && h.b2 < 1.f))
    return fail(VITB200_ERR_INVALID, "adamw_step: b1 and b2 must be in [0, 1)");
  if (!finite(h.eps) || h.eps < 0.f) return fail(VITB200_ERR_INVALID, "adamw_step: eps must be finite and >= 0");
  if (!finite(h.weight_decay) || h.weight_decay < 0.f) return fail(VITB200_ERR_INVALID, "adamw_step: weight_decay must be finite and >= 0");
  if (!finite(h.max_grad_norm) || h.max_grad_norm < 0.f) return fail(VITB200_ERR_INVALID, "adamw_step: max_grad_norm must be finite and >= 0");
  if (!finite(h.grad_scale) || !(h.grad_scale > 0.f)) return fail(VITB200_ERR_INVALID, "adamw_step: grad_scale must be finite and > 0");
  return 0;
}

// moments, status and scratch of the optimiser; the moments start at zero, count at 0
int ensure_optim(vitb200_model* m, cudaStream_t st) {
  auto& ts = *m->train;
  if (ts.status.n) return 0;
  int rc;
  if ((rc = ts.mu.alloc(ts.grads.n)) || (rc = ts.nu.alloc(ts.grads.n)) || (rc = ts.status.alloc(1))) return rc;
  VB_CUDA(cudaMemsetAsync(ts.mu.p, 0, ts.mu.n * sizeof(float), st));
  VB_CUDA(cudaMemsetAsync(ts.nu.p, 0, ts.nu.n * sizeof(float), st));
  VB_CUDA(cudaMemsetAsync(ts.status.p, 0, sizeof(OptStatus), st));
  if (m->fold && (rc = ts.fold_scratch.alloc(fold_scratch_floats(m)))) return rc;
  return 0;
}

// chunks of OPT_CHUNK elements over the trainable leaves; rebuilt when the leaf flags change (stream-ordered upload)
int build_chunk_table(vitb200_model* m, cudaStream_t st) {
  auto& ts = *m->train;
  if (!m->opt_table_dirty && ts.chunks.n) return 0;
  ts.chunks_host.clear();
  for (size_t i = 0; i < m->leaves.size(); ++i) {
    if (!(m->leaf_flags[i] & VITB200_LEAF_TRAINABLE)) continue;
    const int64_t n = m->leaves[i].numel();
    const int32_t decay = (m->leaf_flags[i] & VITB200_LEAF_DECAY) ? 1 : 0;
    for (int64_t s = 0; s < n; s += OPT_CHUNK)
      ts.chunks_host.push_back({m->leaves[i].dev + s, int64_t(ts.grad_off[i]) + s, int32_t(std::min<int64_t>(OPT_CHUNK, n - s)), decay});
  }
  if (!ts.chunks.n) {   // sized once for every leaf trainable: a later change of the flags allocates (and syncs) nothing
    size_t nc = 0;
    for (const auto& l : m->leaves) nc += size_t((l.numel() + OPT_CHUNK - 1) / OPT_CHUNK);
    int rc;
    if ((rc = ts.chunks.alloc(std::max<size_t>(nc, 1))) || (rc = ts.partial.alloc(std::max<size_t>(nc, 1)))) return rc;
  }
  if (!ts.chunks_host.empty())
    VB_CUDA(cudaMemcpyAsync(ts.chunks.p, ts.chunks_host.data(), ts.chunks_host.size() * sizeof(OptChunk), cudaMemcpyHostToDevice, st));
  m->opt_table_dirty = false;
  return 0;
}

// every 16-bit copy the kernels read, re-derived from the fp32 leaves into the same buffers: pointers, tensor maps and
// the captured forward graphs stay valid, and nothing synchronises
int refresh_packed(vitb200_model* m, cudaStream_t st) {
  int rc;
  if ((rc = repack_dense(m, m->patch, st))) return rc;
  for (auto& L : m->layers)
    if ((rc = repack_dense(m, L.qkv, st)) || (rc = repack_dense(m, L.out, st)) || (rc = repack_dense(m, L.ff1, st)) ||
        (rc = repack_dense(m, L.ff2, st))) return rc;
  if (m->head_tc && (rc = repack_dense(m, m->head, st))) return rc;
  if (m->im2col) {
    const auto& c = m->cfg;
    if ((rc = launch_pack_weight_im2col(st, m->leaves[m->patch.leaf_kernel].dev, m->patch_wt_i2c, c.dim, c.patch_h,
                                        c.patch_w * c.channels, m->dt))) return rc;
  }
  if (m->fold) {
    float* scratch = m->train->fold_scratch.p;
    for (auto& L : m->layers)
      if ((rc = refold_dense(m, L.qkv, L.ln1_scale, L.ln1_bias, scratch, st)) ||
          (rc = refold_dense(m, L.ff1, L.ln2_scale, L.ln2_bias, scratch, st))) return rc;
  }
  return 0;
}

}  // namespace

int vitb200_set_leaf_flags(vitb200_model* m, const uint8_t* flags) {
  if (!m || !flags) return fail(VITB200_ERR_INVALID, "set_leaf_flags: null argument");
  for (size_t i = 0; i < m->leaves.size(); ++i)
    if (flags[i] & ~(VITB200_LEAF_TRAINABLE | VITB200_LEAF_DECAY))
      return fail(VITB200_ERR_INVALID, "set_leaf_flags: unknown flag bits for '" + m->leaves[i].path + "'");
  m->leaf_flags.assign(flags, flags + m->leaves.size());
  m->opt_table_dirty = true;
  return 0;
}

int vitb200_adamw_step(vitb200_model* m, void* stream, const vitb200_adamw* h) {
  if (!m || !h) return fail(VITB200_ERR_INVALID, "adamw_step: null argument");
  int rc;
  if ((rc = train_supported(m))) return rc;
  if ((rc = check_adamw(*h))) return rc;
  if (!m->finalized) return fail(VITB200_ERR_PARAM_MISSING, "adamw_step: parameters changed since the backward; call finalize_params");
  if (!m->train || !m->train->grads_fresh)
    return fail(VITB200_ERR_INVALID, "adamw_step: needs a backward with VITB200_GRAD_PARAMS since the last step");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto& ts = *m->train;
  if ((rc = ensure_optim(m, st)) || (rc = build_chunk_table(m, st))) return rc;
  if ((rc = launch_adamw(st, ts.chunks.p, int(ts.chunks_host.size()), ts.grads.p, ts.mu.p, ts.nu.p, ts.partial.p,
                         ts.status.p, *h))) return rc;
  if ((rc = refresh_packed(m, st))) return rc;
  ts.grads_fresh = false;
  ++m->weights_version;
  return 0;
}

int vitb200_optim_status(vitb200_model* m, void* stream, int32_t* count, int32_t* skipped, float* grad_norm) {
  if (!m || !count || !skipped || !grad_norm) return fail(VITB200_ERR_INVALID, "optim_status: null argument");
  *count = 0;
  *skipped = 0;
  *grad_norm = 0.f;
  if (!m->train || !m->train->status.n) return 0;
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  OptStatus s;
  VB_CUDA(cudaMemcpyAsync(&s, m->train->status.p, sizeof(s), cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  *count = s.count;
  *skipped = s.skipped;
  *grad_norm = s.norm;
  return 0;
}

int vitb200_optim_state(vitb200_model* m, float** mu_dev, float** nu_dev, int32_t** count_dev, int64_t* n) {
  if (!m || !mu_dev || !nu_dev || !count_dev || !n) return fail(VITB200_ERR_INVALID, "optim_state: null argument");
  int rc;
  if ((rc = train_supported(m))) return rc;
  if (!m->finalized) return fail(VITB200_ERR_PARAM_MISSING, "optim_state: call finalize_params first");
  DeviceGuard guard(m->device);
  // allocated here, the buffers are zeroed on the legacy stream; the caller may write into them at once from any stream
  // (a checkpoint restored before the first step), so this first-allocation path waits for the zeroing to finish
  const bool fresh = !m->train || !m->train->status.n;
  cudaStream_t st = nullptr;
  if ((rc = ensure_train(m, st)) || (rc = ensure_optim(m, st))) return rc;
  if (fresh) VB_CUDA(cudaStreamSynchronize(st));
  *mu_dev = m->train->mu.p;
  *nu_dev = m->train->nu.p;
  *count_dev = &m->train->status.p->count;
  *n = int64_t(m->train->mu.n);
  return 0;
}

int vitb200_get_param(vitb200_model* m, void* stream, const char* path, float* host_out) {
  if (!m || !path || !host_out) return fail(VITB200_ERR_INVALID, "get_param: null argument");
  auto it = m->index.find(path);
  if (it == m->index.end()) return fail(VITB200_ERR_INVALID, std::string("get_param: unknown parameter path '") + path + "'");
  const Leaf& l = m->leaves[it->second];
  if (!l.set) return fail(VITB200_ERR_PARAM_MISSING, std::string("get_param: parameter '") + path + "' was never set");
  DeviceGuard guard(m->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  VB_CUDA(cudaMemcpyAsync(host_out, l.dev, size_t(l.numel()) * sizeof(float), cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int vitb200_softmax_xent(void* stream, const float* logits, const int32_t* labels, int batch, int classes,
                         float label_smoothing, float dscale, float* loss_dev, float* dlogits_dev) {
  if (!logits || !labels || !loss_dev || !dlogits_dev) return fail(VITB200_ERR_INVALID, "softmax_xent: null pointer");
  if (batch <= 0 || classes <= 0) return fail(VITB200_ERR_INVALID, "softmax_xent: batch and classes must be positive");
  if (!(label_smoothing >= 0.f && label_smoothing <= 1.f)) return fail(VITB200_ERR_INVALID, "softmax_xent: label_smoothing must be in [0, 1]");
  if (!std::isfinite(dscale)) return fail(VITB200_ERR_INVALID, "softmax_xent: dscale must be finite");
  // the kernels and their scratch go to the device that holds the buffers, whichever device is current
  int dev = -1;
  const void* bufs[4] = {logits, labels, loss_dev, dlogits_dev};
  for (const void* b : bufs) {
    cudaPointerAttributes a{};
    VB_CUDA(cudaPointerGetAttributes(&a, b));
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)
      return fail(VITB200_ERR_INVALID, "softmax_xent: logits, labels, loss and dlogits must be device memory");
    if (dev >= 0 && a.device != dev) return fail(VITB200_ERR_INVALID, "softmax_xent: buffers on different devices");
    dev = a.device;
  }
  DeviceGuard guard(dev);
  if (!guard.ok) return fail(VITB200_ERR_CUDA, "softmax_xent: cudaSetDevice failed");
  return launch_softmax_xent(static_cast<cudaStream_t>(stream), logits, labels, batch, classes, label_smoothing, dscale,
                             loss_dev, dlogits_dev);
}

// ---- per-kernel entry points ------------------------------------------------
int vitb200_gemm_tc(void* stream, const void* A, const void* Wt, const float* bias, void* C, int M, int N,
                    int K, int epilogue, const float* aux, int tokens_per_image, int dtype) {
  return vitb200_gemm_tc_dropout(stream, A, Wt, bias, C, M, N, K, epilogue, aux, tokens_per_image, dtype, 0.f, 0, 0);
}

int vitb200_gemm_tc_dropout(void* stream, const void* A, const void* Wt, const float* bias, void* C, int M, int N,
                            int K, int epilogue, const float* aux, int tokens_per_image, int dtype,
                            float rate, uint64_t key, uint32_t site) {
  return vitb200_gemm_tc_tokens(stream, A, Wt, bias, C, M, N, K, epilogue, aux, tokens_per_image, nullptr, dtype,
                                rate, key, site);
}

int vitb200_gemm_tc_tokens(void* stream, const void* A, const void* Wt, const float* bias, void* C, int M, int N,
                           int K, int epilogue, const float* aux, int tokens_per_image, const float* cls, int dtype,
                           float rate, uint64_t key, uint32_t site) {
  if (!(rate >= 0.f && rate < 1.f)) return fail(VITB200_ERR_INVALID, "gemm_tc: dropout rate must be in [0, 1)");
  Dropout drop;
  if (rate > 0.f) {
    drop.key_lo = uint32_t(key);
    drop.key_hi = uint32_t(key >> 32);
    drop.site = site;
    const double t = double(rate) * 4294967296.0;
    drop.threshold = t >= 4294967295.0 ? 0xFFFFFFFFu : uint32_t(t);
    drop.inv_keep = 1.0f / (1.0f - rate);
  }
  if (!A || !Wt || !C) return fail(VITB200_ERR_INVALID, "gemm_tc: null pointer");
  if (M <= 0 || N <= 0 || K <= 0) return fail(VITB200_ERR_INVALID, "gemm_tc: empty problem");
  if ((N % 8) != 0 || (K % 8) != 0)
    return fail(VITB200_ERR_INVALID, "gemm_tc: N and K must be multiples of 8");
  if (dtype != VITB200_DT_BF16 && dtype != VITB200_DT_F16)
    return fail(VITB200_ERR_INVALID, "gemm_tc: dtype must be bf16 or fp16");
  CUtensorMap ta, tb, tc;
  int rc;
  if ((rc = make_tmap_2d(&ta, A, M, K, K, GEMM_BM, dtype))) return rc;
  const int cg = gemm_tc_tile_mode(M, N);
  if ((rc = make_tmap_2d(&tb, Wt, N, K, K, cg == 64 ? 64 : GEMM_BN / cg, dtype))) return rc;
  const bool out16 = epilogue == VITB200_EPI_STORE_16 || epilogue == VITB200_EPI_BIAS_GELU_16 || epilogue == VITB200_EPI_BIAS_16 ||
                     epilogue == VITB200_EPI_BIAS_PRE_GELU_16;
  const bool direct = epilogue == VITB200_EPI_PATCH_F32;
  // PRE_GELU writes its second output tokens_per_image rows below the first: the map covers both
  const int64_t c_rows = epilogue == VITB200_EPI_BIAS_PRE_GELU_16 ? int64_t(tokens_per_image) + M : M;
  if (!direct && (rc = make_tmap_2d(&tc, C, c_rows, N, N, GEMM_BM, out16 ? dtype : VITB200_DT_F32))) return rc;
  return launch_gemm_tc(static_cast<cudaStream_t>(stream), ta, tb, direct ? nullptr : &tc, bias, C, M, N, K, epilogue,
                        aux, tokens_per_image, dtype, cg, drop, 1, cls);
}

int vitb200_patch_embed_im2col(void* stream, const float* images, const float* W, const float* bias, const float* pos,
                               const float* cls, float* x, int batch, int H, int Wd, int C, int ph, int pw, int dim, int dtype,
                               void* x16, float* stats) {
  if (!images || !W || !bias || !pos || !x) return fail(VITB200_ERR_INVALID, "patch_embed_im2col: null pointer");
  if (batch <= 0 || H <= 0 || Wd <= 0 || C <= 0 || ph <= 0 || pw <= 0 || H % ph || Wd % pw)
    return fail(VITB200_ERR_INVALID, "patch_embed_im2col: bad geometry");
  if (!patch_im2col_supported(pw, C, dim))
    return fail(VITB200_ERR_UNSUPPORTED, "patch_embed_im2col: needs pw*C <= 64 floats, a multiple of 16 bytes");
  if ((x16 == nullptr) != (stats == nullptr)) return fail(VITB200_ERR_INVALID, "patch_embed_im2col: x16 and stats go together");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int run = pw * C, kp = ph * 64, gw = Wd / pw, Np = (H / ph) * gw;
  uint16_t* wt = nullptr;
  VB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&wt), size_t(dim) * kp * sizeof(uint16_t), st));
  CUtensorMap tmi, tmw;
  int rc = launch_pack_weight_im2col(st, W, wt, dim, ph, run, dtype);
  if (!rc) rc = make_tmap_2d(&tmw, wt, dim, kp, kp, GEMM_BN, dtype);
  if (!rc) rc = make_tmap_im2col_patches(&tmi, images, batch, H, Wd, C, ph, pw, 128);
  LnFold ln;
  ln.x16 = x16;
  ln.stats = reinterpret_cast<float2*>(stats);
  ln.slots = 2 * ceil_div(dim, GEMM_BN);
  if (!rc && ph > 16) rc = fail(VITB200_ERR_UNSUPPORTED, "patch_embed_im2col: patch height above 16");
  if (!rc) rc = launch_patch_embed_im2col(st, tmi, tmw, bias, pos, cls, x, batch, Np, gw, ph, pw, C, dim, cls ? 1 : 0, dtype,
                                          x16 ? &ln : nullptr);
  cudaFreeAsync(wt, st);
  return rc;
}

int vitb200_gemm_tc_ln_slots(int M, int N) {
  if (M <= 0 || N <= 0) return fail(VITB200_ERR_INVALID, "gemm_tc_ln_slots: empty problem");
  return 2 * ceil_div(N, gemm_tc_tile_mode(M, N) == 64 ? 64 : GEMM_BN);
}

int vitb200_gemm_tc_ln(void* stream, const void* A, const void* Wt, const float* bias, void* C, int M, int N, int K,
                       int epilogue, const float* aux, int tokens_per_image, const float* cls, int dtype,
                       void* x16, float* stats, int stats_slots, const float* ln_c, float ln_eps) {
  if (epilogue < VITB200_EPI_RESID_LN || epilogue > VITB200_EPI_LN_GELU_16)
    return fail(VITB200_ERR_INVALID, "gemm_tc_ln: epilogue must be one of the LayerNorm-fold epilogues (8..11)");
  if (!A || !Wt || !C || !bias || !stats) return fail(VITB200_ERR_INVALID, "gemm_tc_ln: null pointer");
  if (M <= 0 || N <= 0 || K <= 0 || (N % 8) != 0 || (K % 8) != 0)
    return fail(VITB200_ERR_INVALID, "gemm_tc_ln: M, N, K must be positive, N and K multiples of 8");
  if (dtype != VITB200_DT_BF16 && dtype != VITB200_DT_F16) return fail(VITB200_ERR_INVALID, "gemm_tc_ln: dtype must be bf16 or fp16");
  const bool out16 = epilogue == VITB200_EPI_LN_STORE_16 || epilogue == VITB200_EPI_LN_GELU_16;
  const int cg = gemm_tc_tile_mode(M, N);
  CUtensorMap ta, tb, tc;
  int rc;
  if ((rc = make_tmap_2d(&ta, A, M, K, K, GEMM_BM, dtype))) return rc;
  if ((rc = make_tmap_2d(&tb, Wt, N, K, K, cg == 64 ? 64 : GEMM_BN / cg, dtype))) return rc;
  if ((rc = make_tmap_2d(&tc, C, M, N, N, GEMM_BM, out16 ? dtype : VITB200_DT_F32))) return rc;
  LnFold ln;
  ln.x16 = x16;
  ln.stats = reinterpret_cast<float2*>(stats);
  ln.slots = stats_slots;
  ln.c = ln_c;
  ln.eps = ln_eps > 0.f ? ln_eps : 1e-6f;
  return launch_gemm_tc(static_cast<cudaStream_t>(stream), ta, tb, &tc, bias, C, M, N, K, epilogue, aux, tokens_per_image,
                        dtype, cg, Dropout(), 1, cls, ln);
}

int vitb200_fold_layernorm(void* stream, const float* W, const float* gamma, const float* beta, const float* bias,
                           void* Wt, float* c, float* d, int K, int N, int Kpad, int dtype) {
  if (!W || !gamma || !beta || !Wt || !c || !d) return fail(VITB200_ERR_INVALID, "fold_layernorm: null pointer");
  if (K <= 0 || N <= 0 || Kpad < K) return fail(VITB200_ERR_INVALID, "fold_layernorm: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* scratch = nullptr;
  VB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), size_t(K) * N * sizeof(float), st));
  const int rc = launch_fold_layernorm(st, W, gamma, beta, bias, Wt, c, d, K, N, Kpad, dtype, scratch);
  cudaFreeAsync(scratch, st);
  return rc;
}

int vitb200_gemm_tc_e4m3(void* stream, const void* A, const void* Wt, const float* wscale, const float* bias, void* C, int M,
                         int N, int K, int epilogue) {
  if (!A || !Wt || !wscale || !C) return fail(VITB200_ERR_INVALID, "gemm_tc_e4m3: null pointer");
  if (M <= 0 || N <= 0 || K <= 0 || (N % 8) != 0 || (K % 16) != 0)
    return fail(VITB200_ERR_INVALID, "gemm_tc_e4m3: M, N, K must be positive, N a multiple of 8 and K of 16");
  int out_dt;
  switch (epilogue) {
    case VITB200_EPI_STORE_16: out_dt = VITB200_DT_F16; break;
    case VITB200_EPI_BIAS_GELU_E4M3: out_dt = VITB200_DT_E4M3; break;
    case VITB200_EPI_BIAS_RESID_F32: case VITB200_EPI_BIAS_F32: out_dt = VITB200_DT_F32; break;
    default:
      return fail(VITB200_ERR_UNSUPPORTED, "gemm_tc_e4m3: epilogue must be STORE_16, BIAS_GELU_E4M3, BIAS_RESID_F32 or BIAS_F32");
  }
  if (out_dt == VITB200_DT_E4M3 && (N % 16) != 0) return fail(VITB200_ERR_INVALID, "gemm_tc_e4m3: BIAS_GELU_E4M3 needs N % 16 == 0");
  const int cg = gemm_tc_tile_mode(M, N);
  CUtensorMap ta, tb, tc;
  int rc;
  if ((rc = make_tmap_2d(&ta, A, M, K, K, GEMM_BM, VITB200_DT_E4M3))) return rc;
  if ((rc = make_tmap_2d(&tb, Wt, N, K, K, cg == 64 ? 64 : GEMM_BN / cg, VITB200_DT_E4M3))) return rc;
  if ((rc = make_tmap_2d(&tc, C, M, N, N, GEMM_BM, out_dt, out_dt == VITB200_DT_E4M3 ? 64 : 128))) return rc;
  return launch_gemm_tc(static_cast<cudaStream_t>(stream), ta, tb, &tc, bias, C, M, N, K, epilogue, nullptr, 0,
                        VITB200_DT_E4M3, cg, Dropout(), 1, nullptr, LnFold(), wscale);
}

int vitb200_quantize_weight_e4m3(void* stream, const float* W, void* Wt, float* scale, int K, int N, int Kpad) {
  if (!W || !Wt || !scale) return fail(VITB200_ERR_INVALID, "quantize_weight_e4m3: null pointer");
  return launch_quantize_weight_e4m3(static_cast<cudaStream_t>(stream), W, static_cast<uint8_t*>(Wt), scale, K, N, Kpad);
}

int vitb200_gemm_f32(void* stream, const float* A, const float* W, const float* bias, float* C, int M, int N,
                     int K, int epilogue, const float* aux, int tokens_per_image) {
  if (!A || !W || !C) return fail(VITB200_ERR_INVALID, "gemm_f32: null pointer");
  return launch_gemm_f32(static_cast<cudaStream_t>(stream), A, W, bias, C, M, N, K, epilogue, aux, tokens_per_image);
}

int vitb200_layernorm(void* stream, const float* x, const float* scale, const float* bias, void* y, int rows,
                      int dim, int out_dtype) {
  if (!x || !scale || !bias || !y) return fail(VITB200_ERR_INVALID, "layernorm: null pointer");
  return launch_layernorm(static_cast<cudaStream_t>(stream), x, scale, bias, y, rows, dim, out_dtype);
}

int vitb200_attention_tc(void* stream, const void* qkv, void* out, int batch, int T, int heads, int dtype) {
  if (!qkv || !out) return fail(VITB200_ERR_INVALID, "attention_tc: null pointer");
  return launch_attention_tc(static_cast<cudaStream_t>(stream), qkv, out, batch, T, heads, dtype);
}

int vitb200_attention_tc_lse(void* stream, const void* qkv, void* out, float* lse, int batch, int T, int heads, int dtype) {
  if (!qkv || !out || !lse) return fail(VITB200_ERR_INVALID, "attention_tc_lse: null pointer");
  return launch_attention_tc(static_cast<cudaStream_t>(stream), qkv, out, batch, T, heads, dtype, lse);
}

int vitb200_attention_probs(void* stream, const void* qkv, const float* lse, float* maps, int batch, int T, int heads,
                            int dtype) {
  return launch_attention_probs(static_cast<cudaStream_t>(stream), qkv, lse, maps, int64_t(heads) * T * T, batch, T, heads,
                                dtype);
}

int vitb200_attention_f32(void* stream, const float* qkv, float* out, int batch, int T, int heads) {
  if (!qkv || !out) return fail(VITB200_ERR_INVALID, "attention_f32: null pointer");
  return launch_attention_f32(static_cast<cudaStream_t>(stream), qkv, out, batch, T, heads);
}

int vitb200_gemm_tc_wgrad(void* stream, const void* X, const void* dY, float* dW, int M, int N, int K, int splits, int dtype) {
  if (!X || !dY || !dW) return fail(VITB200_ERR_INVALID, "gemm_tc_wgrad: null pointer");
  if (M <= 0 || N <= 0 || K <= 0 || (M % 8) != 0 || (N % 8) != 0)
    return fail(VITB200_ERR_INVALID, "gemm_tc_wgrad: M and N must be positive multiples of 8");
  if (dtype != VITB200_DT_BF16 && dtype != VITB200_DT_F16) return fail(VITB200_ERR_INVALID, "gemm_tc_wgrad: dtype must be bf16 or fp16");
  const int mode = gemm_tc_tile_mode(M, N);
  const int cg = mode == 4 ? 2 : mode;
  CUtensorMap tx, ty, tc;
  int rc;
  if ((rc = make_tmap_2d(&tx, X, K, M, M, 64, dtype))) return rc;
  if ((rc = make_tmap_2d(&ty, dY, K, N, N, 64, dtype))) return rc;
  if ((rc = make_tmap_2d(&tc, dW, M, N, N, GEMM_BM, VITB200_DT_F32))) return rc;
  return launch_gemm_tc_wgrad(static_cast<cudaStream_t>(stream), tx, ty, tc, nullptr, dW, M, N, K, splits, dtype, cg);
}

int vitb200_attention_bwd(void* stream, const void* qkv, const void* out, const void* d_out, void* dqkv, int batch, int T,
                          int heads, int dtype) {
  if (!qkv || !out || !d_out || !dqkv) return fail(VITB200_ERR_INVALID, "attention_bwd: null pointer");
  return launch_attention_bwd(static_cast<cudaStream_t>(stream), qkv, out, d_out, dqkv, batch, T, heads, dtype);
}

int vitb200_layernorm_bwd(void* stream, const void* dy, const float* x, const float* scale, float* dx, float* dscale,
                          float* dbias, int rows, int dim, int dtype, float eps, int accumulate) {
  if (!dy || !x || !scale || !dx || !dscale || !dbias) return fail(VITB200_ERR_INVALID, "layernorm_bwd: null pointer");
  return launch_ln_bwd(static_cast<cudaStream_t>(stream), dy, x, scale, dx, dscale, dbias, rows, dim, dtype,
                       eps > 0.f ? eps : 1e-6f, accumulate);
}

int vitb200_patchify(void* stream, const float* images, void* patches, int batch, int H, int W, int C, int ph,
                     int pw, int Kpad, int out_dtype) {
  if (!images || !patches) return fail(VITB200_ERR_INVALID, "patchify: null pointer");
  return launch_patchify(static_cast<cudaStream_t>(stream), images, patches, batch, H, W, C, ph, pw, Kpad, out_dtype);
}

int vitb200_patchify_tokens(void* stream, const float* images, void* patches, int batch, int H, int W, int C, int ph,
                            int pw, int Kpad, int out_dtype, int nchw, int cls_slot) {
  if (!images || !patches) return fail(VITB200_ERR_INVALID, "patchify: null pointer");
  if ((nchw != 0 && nchw != 1) || (cls_slot != 0 && cls_slot != 1))
    return fail(VITB200_ERR_INVALID, "patchify: nchw and cls_slot are 0 or 1");
  return launch_patchify(static_cast<cudaStream_t>(stream), images, patches, batch, H, W, C, ph, pw, Kpad, out_dtype,
                         nchw, cls_slot);
}

int vitb200_unpatchify(void* stream, const float* patches, float* images, int batch, int H, int W, int C, int ph, int pw,
                       int Kpad, int nchw, int cls_slot) {
  if (!patches || !images) return fail(VITB200_ERR_INVALID, "unpatchify: null pointer");
  if ((nchw != 0 && nchw != 1) || (cls_slot != 0 && cls_slot != 1))
    return fail(VITB200_ERR_INVALID, "unpatchify: nchw and cls_slot are 0 or 1");
  return launch_unpatchify(static_cast<cudaStream_t>(stream), patches, images, batch, H, W, C, ph, pw, Kpad, nchw, cls_slot);
}

int vitb200_cls_rows(void* stream, const float* cls, const float* pos, float* x, int batch, int T, int dim) {
  if (!cls || !pos || !x) return fail(VITB200_ERR_INVALID, "cls_rows: null pointer");
  return launch_cls_rows(static_cast<cudaStream_t>(stream), cls, pos, x, batch, T, dim);
}

int vitb200_pool_layernorm(void* stream, const float* x, const float* scale, const float* bias, void* y,
                           int batch, int T, int dim, int pool, int out_dtype) {
  if (!x || !scale || !bias || !y) return fail(VITB200_ERR_INVALID, "pool_layernorm: null pointer");
  return launch_pool_layernorm(static_cast<cudaStream_t>(stream), x, scale, bias, y, batch, T, dim, pool, out_dtype);
}

int vitb200_pack_weight(void* stream, const float* W, void* Wt, int K, int N, int Kpad, int dtype) {
  if (!W || !Wt) return fail(VITB200_ERR_INVALID, "pack_weight: null pointer");
  if (Kpad < K) return fail(VITB200_ERR_INVALID, "pack_weight: Kpad < K");
  return launch_pack_weight(static_cast<cudaStream_t>(stream), W, Wt, K, N, Kpad, dtype);
}

}  // extern "C"
