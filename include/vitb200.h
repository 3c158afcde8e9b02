/*
 * vitb200.h -- C ABI of the B200-native ViT forward (libvitb200.so).
 *
 * Drop-in boundary for ONE path of conceptofmind/vit-flax: the forward pass of
 * vit_flax/vit.py (ViT.__call__, vit.py:127-167, reached through
 * Module.apply at vit.py:192).  The reference has no FFI seam of its own
 * (SURVEY.md section 8b): its boundary is the Flax Module API.  These entry points are
 * what a jax.ffi / XLA custom-call target (or any ctypes/cgo/JNI binding)
 * would bind for that path; INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, <0 on error; the message for the
 *     calling thread is returned by vitb200_last_error().  Nothing aborts.
 *   - a handle is NOT thread-safe; one handle per (device, stream).
 *   - caller owns image / logits buffers; the library owns packed weights and
 *     the activation workspace (sized for cfg.max_batch images at create).
 *   - no hidden synchronisation in vitb200_forward(): work is enqueued on the
 *     caller's stream.  vitb200_forward_host() is the end-to-end variant with
 *     the H2D / D2H copies and a final stream synchronise.
 *   - there is NO CPU fallback: every compute entry point needs an sm_100a GPU.
 */
#ifndef VITB200_H_
#define VITB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VITB200_ABI_VERSION 4

/* error codes */
#define VITB200_OK                 0
#define VITB200_ERR_INVALID       -1   /* bad argument / shape / config          */
#define VITB200_ERR_CUDA          -2   /* CUDA runtime or driver error           */
#define VITB200_ERR_PARAM_MISSING -3   /* finalize/forward before all params set */
#define VITB200_ERR_UNSUPPORTED   -4   /* valid for the reference, not built yet */
#define VITB200_ERR_NO_DEVICE     -5   /* no sm_100 device visible               */

/* cfg.precision */
#define VITB200_PREC_BF16 0   /* bf16 operands, fp32 accumulate, fp32 residual stream (tcgen05) */
#define VITB200_PREC_FP32 1   /* fp32 everywhere (SIMT validation mode, tolerance 1e-4)        */
#define VITB200_PREC_FP16 2   /* fp16 operands, otherwise identical to BF16 (same tcgen05
                                 kind::f16 rate; 3 more mantissa bits, see DESIGN.md)          */
#define VITB200_PREC_FP8  3   /* inference only: E4M3 operands (tcgen05 kind::f8f6f4) on to_qkv and both
                                 FeedForward Denses -- LayerNorm / GELU outputs unscaled, weights with one
                                 fp32 scale per output column; everything else as FP16.  Dropout > 0 and
                                 every training entry point return VITB200_ERR_UNSUPPORTED (DESIGN.md) */

/* element types of buffers handed to the per-kernel entry points */
#define VITB200_DT_F32  0
#define VITB200_DT_BF16 1
#define VITB200_DT_F16  2
#define VITB200_DT_E4M3 3   /* one byte per element, OCP FP8 E4M3 (max 448, no infinities) */

/* cfg.flags: the variations simple_vit.py needs on the same path (SURVEY.md section 8f-3) */
#define VITB200_FLAG_NCHW   1   /* images are [B, C, H, W] (simple_vit.py:125), not [B, H, W, C]     */
#define VITB200_FLAG_NO_CLS 2   /* no class token: T = num_patches, pos_embedding is [1, Np, dim]   */

/* cfg.pool -- vit.py:121,159 */
#define VITB200_POOL_CLS  0
#define VITB200_POOL_MEAN 1

/* Mirrors the dataclass fields of `class ViT` (vit.py:115-125); dim_head is the
 * reference's class constant 64 (vit.py:123) and is therefore not a field.     */
typedef struct vitb200_config {
  int32_t image_h, image_w;     /* pair(image_size)  vit.py:130 */
  int32_t patch_h, patch_w;     /* pair(patch_size)  vit.py:131 */
  int32_t channels;             /* last axis of x (3 in every reference use) */
  int32_t num_classes;
  int32_t dim;
  int32_t depth;
  int32_t heads;
  int32_t mlp_dim;
  int32_t pool;                 /* VITB200_POOL_*  */
  int32_t precision;            /* VITB200_PREC_*  */
  int32_t max_batch;            /* workspace is sized for this many images   */
  float   dropout;              /* vit.py:124: rate of the Dropouts inside Attention / FeedForward */
  float   emb_dropout;          /* vit.py:125: rate of the Dropout after the positional embedding   */
  int32_t flags;                /* VITB200_FLAG_*; 0 = vit.py                                        */
  float   ln_eps;               /* LayerNorm epsilon; 0 = flax default 1e-6 (vit.py:31,163)          */
  int32_t reserved[1];
} vitb200_config;

typedef struct vitb200_model vitb200_model;   /* opaque */

/* ---- library ---------------------------------------------------------- */
int         vitb200_abi_version(void);
const char* vitb200_last_error(void);
/* number of CUDA devices with compute capability 10.x, or <0 */
int         vitb200_device_count(void);
/* total kernels launched by this library in this process (bench "gpu_launches") */
int64_t     vitb200_launch_count(void);

/* ---- model lifecycle (replaces Module.init/apply plumbing, vit.py:187-192) */
int vitb200_create(const vitb200_config* cfg, int device, vitb200_model** out);
int vitb200_destroy(vitb200_model* m);

/* Number of parameter leaves the config implies and the i-th leaf's path
 * ("Transformer_0/Attention_3/Dense_0/kernel") and shape -- the Flax pytree of
 * SURVEY.md section 8c.  `shape` receives up to 4 dims; returns ndim or <0. */
int vitb200_num_params(const vitb200_model* m);
int vitb200_param_info(const vitb200_model* m, int index, const char** path, int64_t shape[4]);

/* Upload one fp32 leaf (HOST pointer) by path; shape is checked against the
 * config like Flax's ScopeParamShapeError would.                            */
int vitb200_set_param(vitb200_model* m, const char* path, const float* host_data,
                      const int64_t* shape, int ndim);
/* Pack weights for the kernels (bf16 K-major transposes etc.); must be called
 * after all leaves are set and before forward.                              */
int vitb200_finalize_params(vitb200_model* m, void* stream);

/* Key of the 'dropout' rng stream (Flax: rngs={'dropout': key}).  Only used when a rate is > 0:
 * the reference applies every nn.Dropout with deterministic=False (vit.py:50,52,83,155).  The
 * mask of element e of Dropout instance s is Philox4x32-10(key; counter = (e / 4, s)) -- a pure
 * function of the key, like Flax's functional rng (same key => same mask); it cannot be bit-equal
 * to JAX's threefry stream.  Sites: 0 = after pos_embedding; 1+3l = after Attention_l's to_out;
 * 2+3l = after FeedForward_l's GELU; 3+3l = after FeedForward_l's second Dense.               */
int vitb200_set_dropout_key(vitb200_model* m, uint64_t key);

/* ViT.__call__ (vit.py:127-167): images [batch, H, W, C] fp32 NHWC on DEVICE,
 * logits [batch, num_classes] fp32 on DEVICE.  batch <= cfg.max_batch.       */
int vitb200_forward(vitb200_model* m, void* stream, const float* images_dev, int batch,
                    float* logits_dev);
/* Same call with HOST buffers (pinned or pageable): H2D, forward, D2H, sync. */
int vitb200_forward_host(vitb200_model* m, void* stream, const float* images_host, int batch,
                         float* logits_host);
/* Pipelined end-to-end variant for a stream of batches: submit enqueues H2D (own copy stream),
 * forward (caller's stream) and D2H (own copy stream) of one batch and returns at once; at most
 * two jobs may be in flight, so the H2D copy of batch k+1 overlaps the forward of batch k.
 * wait_host blocks until the OLDEST submitted job's logits are in `logits_host`.  Host buffers
 * should be pinned and must stay valid until the job has been waited for.                     */
/* vitb200_forward that also records the attention weights softmax(Q K^T * 64^-0.5) (vit.py:73-75) of the layers
 * layers[0 .. n_layers) (HOST array of distinct indices in [0, depth), any order) into maps_dev, fp32 on DEVICE,
 * [batch, n_layers, heads, T, T] in that order (T counts the class token; vit-pytorch's Recorder layout).  The logits
 * are those of vitb200_forward; unrecorded layers run what vitb200_forward runs.  A recorded layer passes a row
 * log-sum-exp buffer to its attention kernel and recomputes P from the same 16-bit q / k right after it, on tcgen05.
 * Never replays or captures the forward graphs.  The first call allocates a [max_batch * heads, T] fp32 scratch kept
 * with the model.  fp32 models: VITB200_ERR_UNSUPPORTED.                                                           */
int vitb200_forward_attn(vitb200_model* m, void* stream, const float* images_dev, int batch, float* logits_dev,
                         const int* layers, int n_layers, float* maps_dev);
int vitb200_submit_host(vitb200_model* m, void* stream, const float* images_host, int batch,
                        float* logits_host);
int vitb200_wait_host(vitb200_model* m);
/* One forward with a CUDA event before every launch: per-category device time (ms) and launch
 * counts, arrays of VITB200_NUM_CATEGORIES.  Synchronises the stream.  For bench/roofline.  */
#define VITB200_CAT_PATCHIFY   0
#define VITB200_CAT_GEMM_PATCH 1
#define VITB200_CAT_CLS_ROWS   2
#define VITB200_CAT_LAYERNORM  3
#define VITB200_CAT_GEMM_QKV   4
#define VITB200_CAT_ATTENTION  5
#define VITB200_CAT_GEMM_OUT   6
#define VITB200_CAT_GEMM_FF1   7
#define VITB200_CAT_GEMM_FF2   8
#define VITB200_CAT_POOL_LN    9
#define VITB200_CAT_GEMM_HEAD  10
#define VITB200_NUM_CATEGORIES 11
int vitb200_profile_forward(vitb200_model* m, void* stream, const float* images_dev, int batch,
                            float* logits_dev, float* ms_by_category, int* launches_by_category);
/* Copy the token stream after the last block ([batch, T, dim] fp32, device to
 * host) -- parity checks of Transformer.__call__ (vit.py:98-112).  A dropout-free
 * tcgen05 forward with pool = cls computes the last block for the class-token rows
 * only (DESIGN.md section 3, class-token tail): after such a forward this returns
 * VITB200_ERR_UNSUPPORTED rather than stale rows.  A forward that records the last
 * layer (vitb200_forward_attn), mean pooling, dropout > 0 and fp32 models run the
 * whole block, and the stream is readable after them.                          */
int vitb200_debug_tokens(vitb200_model* m, void* stream, float* tokens_host, int batch);

/* ---- training: forward that keeps its activations + backward (SURVEY.md section 8f-4) -----
 * Nothing in the reference trains (no jax.grad anywhere in vit_flax), so these have no reference
 * counterpart; they are the two halves of jax.vjp(lambda p: ViT.apply(p, img), params).
 * Built for the bf16 / fp16 modes and dim <= 1280; anything else returns VITB200_ERR_UNSUPPORTED.  With dropout rates > 0 the forward draws its masks from the key of
 * vitb200_set_dropout_key and the backward replays them (they are pure functions of key, site, element).  Activations (about 5.4 KB per token and layer for
 * ViT-B) and one fp32 gradient per leaf are allocated for max_batch on the first call.           */
int vitb200_train_forward(vitb200_model* m, void* stream, const float* images_dev, int batch,
                          float* logits_dev);
/* dlogits_dev: [batch, num_classes] fp32, the cotangent of the logits of the last train_forward.
 * 16-bit intermediates: with fp16 operands scale dlogits up (and the gradients down) yourself
 * when its entries are below ~1e-4 (loss scaling); gradients are linear in dlogits.             */
int vitb200_backward(vitb200_model* m, void* stream, const float* dlogits_dev, int batch);
/* What a backward differentiates with respect to (jax.vjp(v.apply, params, x) takes both): */
#define VITB200_GRAD_PARAMS 1   /* one fp32 gradient per parameter leaf (vitb200_get_grad & co.)  */
#define VITB200_GRAD_IMAGES 2   /* the gradient of the images given to train_forward            */
/* wrt: a non-zero OR of the two flags.  dimages_dev: required iff VITB200_GRAD_IMAGES; fp32, the layout of the images
 * given to train_forward ([B,H,W,C], or [B,C,H,W] for VITB200_FLAG_NCHW models), fully overwritten.  Image gradients are
 * the same bits with or without VITB200_GRAD_PARAMS.  Without it the weight-gradient GEMMs are skipped (saliency /
 * adversarial loops want dimages only) and vitb200_get_grad, vitb200_grad_device and vitb200_grads_buffer return
 * VITB200_ERR_INVALID until a backward with VITB200_GRAD_PARAMS runs.  The first image-gradient backward allocates a
 * [max_batch * T, round_up(ph*pw*C, 64)] fp32 scratch (patch-feature gradients) kept with the model.
 * vitb200_backward(m, s, dl, b) == vitb200_backward_ex(m, s, dl, b, VITB200_GRAD_PARAMS, NULL).                    */
int vitb200_backward_ex(vitb200_model* m, void* stream, const float* dlogits_dev, int batch,
                        int wrt, float* dimages_dev);
/* gradient of one leaf (flax path, same shape as the parameter) -> host; synchronises the stream */
int vitb200_get_grad(vitb200_model* m, void* stream, const char* path, float* host_out);
/* all leaf gradients as ONE contiguous fp32 buffer (leaves 256-byte aligned, padding zero): the unit of
 * the data-parallel gradient all-reduce -- one collective per step instead of one per leaf            */
int vitb200_grads_buffer(vitb200_model* m, float** dev_out, int64_t* count);
/* device pointer of the same gradient (valid until the model is destroyed; overwritten by backward) */
int vitb200_grad_device(vitb200_model* m, const char* path, float** dev_out);

/* ---- on-device training step: AdamW on the fp32 leaves, then the 16-bit copies re-derived in place ----------------
 * Semantics of optax.apply_if_finite(optax.chain(optax.clip_by_global_norm(max_grad_norm), optax.adamw(...))) with the
 * gradient g = grads_buffer * grad_scale * clip, t = count + 1:
 *   mu = b1 mu + (1 - b1) g;  nu = b2 nu + (1 - b2) g^2;  p -= lr ((mu / (1 - b1^t)) / (sqrt(nu / (1 - b2^t)) + eps) + wd p)
 * (the weight-decay term only on DECAY leaves).  clip = max_grad_norm / max(norm, max_grad_norm), or 1 when
 * max_grad_norm is 0; norm = the global norm of g over the TRAINABLE leaves.  When any such gradient is not finite the
 * step is skipped: parameters, mu, nu and count stay bit for bit as they were and `skipped` reads 1.             */
typedef struct vitb200_adamw {
  float lr, b1, b2, eps, weight_decay;
  float max_grad_norm;   /* 0 = no clipping (optax.clip_by_global_norm)                         */
  float grad_scale;      /* multiplies the gradient buffer: 1 / (loss scale * data-parallel world) */
  int32_t reserved[4];
} vitb200_adamw;
#define VITB200_LEAF_TRAINABLE 1   /* the leaf is updated (a frozen leaf is never read or written by the step) */
#define VITB200_LEAF_DECAY     2   /* the weight-decay term applies (optax.adamw's mask)                      */
/* num_params entries in param_info order; default: every leaf TRAINABLE | DECAY (optax.adamw without a mask) */
int vitb200_set_leaf_flags(vitb200_model* m, const uint8_t* flags);
/* Asynchronous (no host synchronisation): the gradient norm, the update and the re-derivation of every packed 16-bit
 * weight copy (transposed packs, Flax-layout copies, LayerNorm folds) from the new fp32 leaves INTO THE SAME BUFFERS,
 * so the captured small-batch forward graphs stay valid.  Needs a vitb200_backward_ex with VITB200_GRAD_PARAMS since
 * the last step (else VITB200_ERR_INVALID); afterwards a backward whose train_forward ran before the step is refused.
 * mu / nu (fp32, the layout of vitb200_grads_buffer) and the fold scratch are allocated by the first step.
 * vitb200_set_param / vitb200_finalize_params do not touch mu, nu or count.  fp32 models: VITB200_ERR_UNSUPPORTED. */
int vitb200_adamw_step(vitb200_model* m, void* stream, const vitb200_adamw* h);
/* count, skipped and grad_norm (the norm of the last step, NaN when it was skipped); synchronises the stream */
int vitb200_optim_status(vitb200_model* m, void* stream, int32_t* count, int32_t* skipped, float* grad_norm);
/* device pointers of mu, nu ([n] fp32 each; leaf i at element offset sum_{j<i} round_up(numel_j, 64), padding zero) and
 * of count (int32), for checkpoints and resumption; allocates them (zero) if no step has run yet, and then waits for the
 * zeroing to finish, so the caller may write into them from any stream */
int vitb200_optim_state(vitb200_model* m, float** mu_dev, float** nu_dev, int32_t** count_dev, int64_t* n);
/* one fp32 parameter leaf (flax path) -> host; synchronises the stream */
int vitb200_get_param(vitb200_model* m, void* stream, const char* path, float* host_out);
/* optax.softmax_cross_entropy(logits, optax.smooth_labels(one_hot(labels), label_smoothing)).mean() and its gradient
 * in one pass: logits [batch, classes] fp32, labels [batch] int32 (all DEVICE pointers) -> *loss_dev (fp32, reduced in
 * a fixed order) and dlogits_dev = dscale * d loss / d logits.  A label outside [0, classes) makes the loss and its row
 * of dlogits NaN (a following vitb200_adamw_step then skips).  All four buffers must be on one device; the kernels run
 * there whatever device is current, and `stream` must belong to it.                                                */
int vitb200_softmax_xent(void* stream, const float* logits, const int32_t* labels, int batch, int classes,
                         float label_smoothing, float dscale, float* loss_dev, float* dlogits_dev);

/* ---- per-kernel entry points (unit parity tests, ncu) -------------------
 * All pointers are DEVICE pointers.                                         */

/* gemm epilogues ("16" = the 16-bit operand type of the call, bf16 or fp16) */
#define VITB200_EPI_STORE_16        0  /* C_16 = acc                           (to_qkv, vit.py:68)   */
#define VITB200_EPI_BIAS_GELU_16    1  /* C_16 = gelu_tanh(acc + bias)         (vit.py:48-49)        */
#define VITB200_EPI_BIAS_RESID_F32  2  /* C_f32 += acc + bias  (in place)      (vit.py:51/82 + 39)   */
#define VITB200_EPI_BIAS_F32        3  /* C_f32 = acc + bias                   (head, vit.py:165)    */
#define VITB200_EPI_PATCH_F32       4  /* C_f32[b*T+1+t] = acc + bias + pos[1+t]  (vit.py:147-153)   */
#define VITB200_EPI_TOKENS_F32      5  /* A in token layout (row b*T+t; t = 0 the class-token slot):
                                        * C_f32[b*T+t] = t == 0 && cls ? cls + pos[0]
                                        *                              : acc + bias + pos[t]  (vit.py:147-153) */
#define VITB200_EPI_BIAS_16         6  /* C_16 = acc + bias  (FF pre-activation kept for the backward pass) */
#define VITB200_EPI_BIAS_PRE_GELU_16 7 /* two outputs in one [2*off, N] buffer: C_16[r] = pre = acc + bias and
                                        * C_16[r + off] = gelu_tanh(pre), off = tokens_per_image >= M, a multiple of
                                        * 256 (training forward: FF Dense_0 without a separate GELU pass)        */

/* LayerNorm fold (PreNorm, vit.py:31): LN(x) W = rstd (x W') - rstd mean c + d,  W' = diag(gamma) W, c = 1^T W',
 * d = beta^T W (+ bias).  The two GEMMs that PRODUCE the residual stream also emit what the next LayerNorm needs, the
 * two that CONSUME a LayerNorm apply it in their epilogue: no stand-alone LayerNorm kernel in between.  Only through
 * vitb200_gemm_tc_ln.                                                                                                */
#define VITB200_EPI_RESID_LN        8  /* C_f32 = C_f32 + acc + bias (x_old read by TMA, added in the SM, stored back);
                                        * x16[M,N] = 16-bit copy of C; stats[M, slots] = per-row partial (sum, sum sq)   */
#define VITB200_EPI_TOKENS_LN       9  /* EPI_TOKENS_F32 + the same x16 / stats outputs (patch embedding, vit.py:147-153) */
#define VITB200_EPI_LN_STORE_16     10 /* C_16 = rstd*acc - rstd*mean*c + d        (to_qkv after PreNorm, vit.py:31,68)    */
#define VITB200_EPI_LN_GELU_16      11 /* C_16 = gelu_tanh(rstd*acc - rstd*mean*c + d)  (FeedForward Dense_0, vit.py:48-49) */
#define VITB200_EPI_BIAS_GELU_E4M3  12 /* C_e4m3 = satfinite(e4m3(gelu_tanh(acc*wscale + bias)))  (fp8 FeedForward Dense_0)  */

/* tcgen05 GEMM: acc[M,N] = A[M,K] (16-bit row-major) x Wt[N,K]^T (16-bit row-major, i.e. the
 * transposed Flax kernel), fp32 accumulation in TMEM.  dtype = VITB200_DT_BF16 | _F16.
 * K % 8 == 0, N % 8 == 0.  `aux` = pos_embedding [T, N] fp32 and `tokens_per_image` = T-1 for
 * EPI_PATCH.  For EPI_BIAS_RESID_F32, `tokens_per_image` > 1 is a split-K factor: that many CTAs
 * share a tile's K range and their partial sums meet in the reduce-add (used by the weight-gradient
 * GEMMs, whose outputs have few tiles and a very long K).                                       */
int vitb200_gemm_tc(void* stream, const void* A, const void* Wt, const float* bias,
                    void* C, int M, int N, int K, int epilogue,
                    const float* aux, int tokens_per_image, int dtype);
/* Same with the Dropout that follows the Dense in the reference (epilogues 1, 2, 4 and 5 only):
 * rate in [0, 1), key / site as in vitb200_set_dropout_key.                                   */
int vitb200_gemm_tc_dropout(void* stream, const void* A, const void* Wt, const float* bias,
                            void* C, int M, int N, int K, int epilogue,
                            const float* aux, int tokens_per_image, int dtype,
                            float rate, uint64_t key, uint32_t site);
/* Same with the class-token row source of EPI_TOKENS (`cls` [N] fp32 or NULL; ignored by the other
 * epilogues except EPI_PATCH, where a non-NULL cls also writes row b*T = cls + pos[0]).
 * For EPI_TOKENS `tokens_per_image` = T (rows per image of A and C) and `aux` = pos_embedding [T, N]. */
int vitb200_gemm_tc_tokens(void* stream, const void* A, const void* Wt, const float* bias,
                           void* C, int M, int N, int K, int epilogue,
                           const float* aux, int tokens_per_image, const float* cls, int dtype,
                           float rate, uint64_t key, uint32_t site);
/* The patch embedding as ONE kernel (vit.py:146-153; csrc/patch_tc.cu): im2col-mode TMA over NHWC fp32 images (no patch
 * matrix in memory) + tcgen05 GEMM + bias + pos_embedding + class-token rows.  W: the Flax kernel [ph*pw*C, dim] fp32
 * (packed inside; the model path packs once), pos [T, dim], cls [dim] or NULL (no class token: T = Np), x [batch*T, dim]
 * fp32 out.  x16 / stats (both or neither): the LayerNorm-fold outputs, stats [batch*T, 2*ceil(dim/256)] float pairs.
 * Needs pw*C <= 64 and pw*C*4 a multiple of 16 bytes (every /16 patch size); else VITB200_ERR_UNSUPPORTED.            */
int vitb200_patch_embed_im2col(void* stream, const float* images, const float* W, const float* bias,
                               const float* pos, const float* cls, float* x, int batch, int H, int W_px, int C,
                               int ph, int pw, int dim, int dtype, void* x16, float* stats);

/* The LayerNorm-fold epilogues (8..11).  Producers (8, 9): `x16` [M,N] 16-bit and `stats` [M, stats_slots] float pairs
 * are OUTPUTS, stats_slots = 2 * ceil(N / tile columns) (tile columns: 256, or 64 when M <= 256 and N > 256 -- ask
 * vitb200_gemm_tc_ln_slots).  Consumers (10, 11): `stats` / `stats_slots` are those of the GEMM that produced A's rows
 * (its N == this K), `ln_c` [N] the column sums c, `bias` the vector d [N] (vitb200_fold_layernorm makes W', c, d),
 * `ln_eps` the LayerNorm epsilon; A is the producer's x16.  No dropout variants.                                        */
int vitb200_gemm_tc_ln(void* stream, const void* A, const void* Wt, const float* bias,
                       void* C, int M, int N, int K, int epilogue,
                       const float* aux, int tokens_per_image, const float* cls, int dtype,
                       void* x16, float* stats, int stats_slots, const float* ln_c, float ln_eps);
int vitb200_gemm_tc_ln_slots(int M, int N);
/* W fp32 [K,N] (Flax kernel), gamma / beta [K] (LayerNorm scale / bias), bias [N] or NULL ->
 * Wt 16-bit [N,Kpad] = (diag(gamma) W)^T, c [N] = column sums of the ROUNDED W', d [N] = beta^T W + bias            */
int vitb200_fold_layernorm(void* stream, const float* W, const float* gamma, const float* beta, const float* bias,
                           void* Wt, float* c, float* d, int K, int N, int Kpad, int dtype);
/* fp8 tcgen05 GEMM (kind::f8f6f4): acc[M,N] = A[M,K] x Wt[N,K]^T with A and Wt E4M3 codes (row-major, K % 16 == 0 so
 * that a row is a legal 16-byte TMA pitch), fp32 accumulation; every epilogue first multiplies acc by wscale[n] (the
 * per-column weight scale of vitb200_quantize_weight_e4m3).  epilogue: STORE_16 (C fp16 = acc*wscale), BIAS_GELU_E4M3
 * (C E4M3, N % 16 == 0), BIAS_RESID_F32 (C fp32 += acc*wscale + bias) or BIAS_F32 (C fp32 = acc*wscale + bias).      */
int vitb200_gemm_tc_e4m3(void* stream, const void* A, const void* Wt, const float* wscale, const float* bias,
                         void* C, int M, int N, int K, int epilogue);
/* W fp32 [K,N] (Flax kernel) -> Wt E4M3 [N,Kpad] (K-major, zero for k >= K; Kpad % 16 == 0) and scale [N] fp32:
 * scale[n] = max_k |W[k,n]| / 448 (1 for an all-zero column), Wt[n,k] = satfinite(e4m3(W[k,n] / scale[n])), rounded
 * to nearest even.                                                                                                   */
int vitb200_quantize_weight_e4m3(void* stream, const float* W, void* Wt, float* scale, int K, int N, int Kpad);
/* SIMT fp32 GEMM (validation mode): acc = A[M,K] x W[K,N] (Flax layout).
 * The two "_16" epilogues write fp32 here.                                  */
int vitb200_gemm_f32(void* stream, const float* A, const float* W, const float* bias,
                     float* C, int M, int N, int K, int epilogue,
                     const float* aux, int tokens_per_image);

/* nn.LayerNorm() (vit.py:31,163): x [rows, dim] fp32 -> y of type out_dtype (VITB200_DT_*; E4M3 = satfinite(e4m3(.)),
 * round to nearest even, the A operand of the fp8 GEMMs) */
int vitb200_layernorm(void* stream, const float* x, const float* scale, const float* bias,
                      void* y, int rows, int dim, int out_dtype);

/* softmax(Q K^T * 64^-0.5) V per (image, head) (vit.py:69-79).  qkv is the
 * to_qkv output [batch*T, 3*heads*64] (q | k | v, head-major inside each),
 * out is [batch*T, heads*64].  _tc = flash-style tensor-core kernel on 16-bit data. */
int vitb200_attention_tc(void* stream, const void* qkv, void* out, int batch, int T, int heads,
                         int dtype);
/* The same kernel, also writing lse [batch*heads, T] fp32 = log2 sum_j exp2(s_ij * 64^-0.5 * log2(e)), the row
 * log-sum-exp in the log2 domain (row b*heads + h, column i); `out` is the same bits as vitb200_attention_tc's. */
int vitb200_attention_tc_lse(void* stream, const void* qkv, void* out, float* lse, int batch, int T, int heads,
                             int dtype);
/* The attention weights alone: maps [batch, heads, T, T] fp32 = exp2(s_ij * 64^-0.5 * log2(e) - lse_i) with s = q k^T
 * of the 16-bit qkv and lse from vitb200_attention_tc_lse on the same qkv.  Every element inside [T, T] is written. */
int vitb200_attention_probs(void* stream, const void* qkv, const float* lse, float* maps, int batch, int T, int heads,
                            int dtype);
int vitb200_attention_f32(void* stream, const float* qkv, float* out, int batch, int T, int heads);

/* weight gradient dW[M, N] += X[K, M]^T dY[K, N]: X and dY are the row-major 16-bit activations
 * (K = rows, any count; M, N % 8 == 0), read as MN-major tcgen05 operands; `splits` CTAs share a
 * tile's K range (<= 1: none) and meet in the fp32 reduce-add.  dW must be initialised (it accumulates). */
int vitb200_gemm_tc_wgrad(void* stream, const void* X, const void* dY, float* dW,
                          int M, int N, int K, int splits, int dtype);
/* adjoint of vitb200_attention_tc: (qkv, out = the forward's output, d_out [batch*T, heads*64])
 * -> dqkv [batch*T, 3*heads*64]; T <= 208 runs one shared-memory-resident kernel, larger T the streamed kernels
 * (with stream-ordered scratch here; the model path owns its workspace) */
int vitb200_attention_bwd(void* stream, const void* qkv, const void* out, const void* d_out, void* dqkv,
                          int batch, int T, int heads, int dtype);
/* adjoint of vitb200_layernorm: dx (+)= d/dx, dscale += , dbias += ; dy is 16-bit of `dtype`, dim <= 1280 */
int vitb200_layernorm_bwd(void* stream, const void* dy, const float* x, const float* scale,
                          float* dx, float* dscale, float* dbias, int rows, int dim, int dtype,
                          float eps, int accumulate);
/* The same with the outputs the training backward fuses into it.  dx (fp32) is stored WITHOUT the mask.  dx16 (NULL or
 * [rows, dim] of `dtype`) = the new dx with the Dropout mask (rate, key, site; as in vitb200_gemm_tc_dropout, flat index
 * r * dim + c) applied in fp32, rounded once; dbias_next (NULL, or non-NULL only with dx16) += column sums of those masked
 * fp32 values.  vitb200_layernorm_bwd(...) == vitb200_layernorm_bwd_ex(..., NULL, NULL, 0, 0, 0).                */
int vitb200_layernorm_bwd_ex(void* stream, const void* dy, const float* x, const float* scale,
                             float* dx, float* dscale, float* dbias, int rows, int dim, int dtype,
                             float eps, int accumulate, void* dx16, float* dbias_next,
                             float rate, uint64_t key, uint32_t site);
/* Bias-gradient row passes (cols % 8 == 0; the Dropout triple as above, replayed on the flat index r * cols + c):
 * cast16_colsum:   y16 = round(Dropout(x)),                          sums[c] += sum_r Dropout(x)[r, c]   (fp32 values)
 * gelu_bwd_colsum: dpre16 = round(Dropout(dhid16 * gelu_tanh'(pre16))), sums[c] += sum_r dpre16[r, c]   (ROUNDED values)
 * gelu' uses tanh.approx (2^-11 relative).  dpre may be dhid (in place).  sums accumulate.                           */
int vitb200_cast16_colsum(void* stream, const float* x, void* y16, float* sums, int rows, int cols, int dtype,
                          float rate, uint64_t key, uint32_t site);
int vitb200_gelu_bwd_colsum(void* stream, const void* pre, const void* dhid, void* dpre, float* sums, int rows,
                            int cols, int dtype, float rate, uint64_t key, uint32_t site);
/* hid16 = round(Dropout(gelu_tanh(pre16))) over n elements (n % 8 == 0, flat index i): the FF activation of a training
 * forward that keeps the GELU out of the GEMM epilogue (VITB200_TRAIN_DUAL=0)                                     */
int vitb200_gelu_fwd(void* stream, const void* pre, void* hid, int64_t n, int dtype, float rate, uint64_t key,
                     uint32_t site);
/* x = Dropout(x) in place, fp32, n % 4 == 0 (the embedding dropout's mask in the backward pass); rate 0: nothing */
int vitb200_dropout_inplace(void* stream, float* x, int64_t n, float rate, uint64_t key, uint32_t site);
/* Adjoint of vitb200_pool_layernorm (fp32; pool 0 = cls, 1 = mean): x [batch, T, dim] the pooled input, dy [batch, dim]
 * the cotangent of the LayerNorm output -> dpooled [batch, dim] = the gradient of one token row (cls: of row 0; mean: of
 * every row, i.e. the pooled gradient / T), dx [batch, T, dim] fully overwritten (cls: zero rows for t > 0), dscale /
 * dbias +=.  dim % 4 == 0.  dpooled may be dy.                                                                      */
int vitb200_pool_layernorm_bwd(void* stream, const float* x, const float* dy, const float* scale, float* dpooled,
                               float* dx, float* dscale, float* dbias, int batch, int T, int dim, int pool, float eps);
/* Head Dense backward (fp32): pooled [batch, dim], dlogits [batch, classes], W [dim, classes] (Flax kernel) ->
 * dpooled [batch, dim] = dlogits W^T (overwritten); dW (NULL: skipped) += pooled^T dlogits; dbias (NULL: skipped) +=
 * column sums of dlogits.                                                                                          */
int vitb200_head_bwd(void* stream, const float* pooled, const float* dlogits, const float* W, float* dW, float* dbias,
                     float* dpooled, int batch, int dim, int classes);
/* Token-embedding gradients (vit.py:151-153) from dx [batch, T, dim] fp32: dpos [T, dim] = sum_b dx[b].  dpos MUST be
 * zero on entry: its sums are written with plain adds and then read back for the others.  cls_slot 1: dcls [dim] +=
 * dpos[0], dbias [dim] += sum_{t >= 1} dpos[t]; cls_slot 0: dbias += sum_t dpos[t], dcls unused (may be NULL).      */
int vitb200_token_grads(void* stream, const float* dx, float* dpos, float* dcls, float* dbias, int batch, int T,
                        int dim, int cls_slot);

/* patchify (vit.py:146): images [batch,H,W,C] fp32 -> patches [batch*Np, Kpad] of out_dtype,
 * feature f = (p1*pw + p2)*C + c, zero padded to Kpad. */
int vitb200_patchify(void* stream, const float* images, void* patches, int batch,
                     int H, int W, int C, int ph, int pw, int Kpad, int out_dtype);
/* Same with the image layout (nchw = 1: [batch,C,H,W], simple_vit.py:125) and the token layout of
 * the forward (cls_slot = 1: patch t of image b goes to row b*(Np+1) + 1 + t; row b*(Np+1), the
 * class-token slot consumed by EPI_TOKENS, is left untouched). */
int vitb200_patchify_tokens(void* stream, const float* images, void* patches, int batch,
                            int H, int W, int C, int ph, int pw, int Kpad, int out_dtype,
                            int nchw, int cls_slot);
/* adjoint of vitb200_patchify_tokens with fp32 patches (the last step of an image-gradient backward):
 * patches [batch*(Np+cls_slot), Kpad] fp32 -> images fp32 in the layout `nchw` selects.  A pure permutation: every
 * pixel is written once; the pad columns and the class-token slot rows are not read. */
int vitb200_unpatchify(void* stream, const float* patches, float* images, int batch, int H, int W,
                       int C, int ph, int pw, int Kpad, int nchw, int cls_slot);
/* cls rows (vit.py:151-153): x[b*T + 0, :] = cls + pos[0] */
int vitb200_cls_rows(void* stream, const float* cls, const float* pos, float* x,
                     int batch, int T, int dim);
/* pool (vit.py:159) + head LayerNorm (vit.py:163): x [batch,T,dim] fp32 -> y [batch, dim] */
int vitb200_pool_layernorm(void* stream, const float* x, const float* scale, const float* bias,
                           void* y, int batch, int T, int dim, int pool, int out_dtype);
/* fp32 [K,N] (Flax kernel) -> 16-bit [N,Kpad] transposed pack used by gemm_tc */
int vitb200_pack_weight(void* stream, const float* W, void* Wt, int K, int N, int Kpad, int dtype);

#ifdef __cplusplus
}
#endif
#endif /* VITB200_H_ */
