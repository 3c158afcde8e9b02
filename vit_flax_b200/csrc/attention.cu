// attention.cu -- entry point of the fused attention  out = softmax(Q K^T * 64^-0.5) V  (vit.py:69-79).
//
// Both kernels are tcgen05 / TMEM ones: attention_tc5.cu when the keys of an (image, head) fit one block (T <= 208: every
// 224-px /16 config), attention_tc5m.cu with streamed key blocks and an online softmax beyond (ViT-H/14: 257 tokens,
// 512 px: 1025).  The first generation of this file -- warp-level mma.sync with a streamed-KV online softmax, 155 / 1551 us
// against 81 / 814 us at T = 257 / 1025 (profiles/r01_attention.md) -- was the baseline the tcgen05 kernels were measured
// against; it was removed at the end of round 2 (git history: attention.cu before "mma.sync generation removed").
#include "common.h"
#include "ptx.cuh"

namespace vb {

int launch_attention_tc(cudaStream_t stream, const void* qkv, void* out, int batch, int T, int heads,
                        int dtype, float* lse, int q_tiles) {
  if (batch <= 0 || T <= 0 || heads <= 0)
    return fail(VITB200_ERR_INVALID, "attention_tc: empty problem");
  if (attention_tc5_supports(T)) return launch_attention_tc5(stream, qkv, out, batch, T, heads, dtype, lse, q_tiles);
  return launch_attention_tc5m(stream, qkv, out, batch, T, heads, dtype, lse, q_tiles);
}

}  // namespace vb
