"""ctypes binding of ``libvitb200.so`` (the C ABI declared in ``include/vitb200.h``).

There is no CPU fallback: if the shared object is missing, ``load()`` raises.
Build it with ``python -m vit_flax_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libvitb200.so"

# error codes / enums (keep in sync with include/vitb200.h)
ABI_VERSION = 4
FLAG_NCHW, FLAG_NO_CLS = 1, 2
OK = 0
PREC_BF16, PREC_FP32, PREC_FP16, PREC_FP8 = 0, 1, 2, 3
DT_F32, DT_BF16, DT_F16, DT_E4M3 = 0, 1, 2, 3
PRECISIONS = {"bf16": PREC_BF16, "fp32": PREC_FP32, "fp16": PREC_FP16, "fp8": PREC_FP8}
POOL_CLS, POOL_MEAN = 0, 1
CATEGORIES = ["patchify", "gemm_patch", "cls_rows", "layernorm", "gemm_qkv", "attention", "gemm_out",
              "gemm_ff1", "gemm_ff2", "pool_ln", "gemm_head"]
EPI_STORE_16, EPI_BIAS_GELU_16, EPI_BIAS_RESID_F32, EPI_BIAS_F32, EPI_PATCH_F32, EPI_TOKENS_F32, EPI_BIAS_16, EPI_BIAS_PRE_GELU_16 = range(8)
EPI_RESID_LN, EPI_TOKENS_LN, EPI_LN_STORE_16, EPI_LN_GELU_16 = range(8, 12)
EPI_BIAS_GELU_E4M3 = 12
GRAD_PARAMS, GRAD_IMAGES = 1, 2
LEAF_TRAINABLE, LEAF_DECAY = 1, 2


class Config(C.Structure):
    _fields_ = [
        ("image_h", C.c_int32), ("image_w", C.c_int32),
        ("patch_h", C.c_int32), ("patch_w", C.c_int32),
        ("channels", C.c_int32), ("num_classes", C.c_int32),
        ("dim", C.c_int32), ("depth", C.c_int32), ("heads", C.c_int32),
        ("mlp_dim", C.c_int32), ("pool", C.c_int32), ("precision", C.c_int32),
        ("max_batch", C.c_int32), ("dropout", C.c_float), ("emb_dropout", C.c_float),
        ("flags", C.c_int32), ("ln_eps", C.c_float), ("reserved", C.c_int32 * 1),
    ]


class AdamW(C.Structure):
    _fields_ = [("lr", C.c_float), ("b1", C.c_float), ("b2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("max_grad_norm", C.c_float), ("grad_scale", C.c_float),
                ("reserved", C.c_int32 * 4)]


class VitB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"vitb200 error {code}: {message}")
        self.code = code
        self.message = message


_vp, _i, _i64 = C.c_void_p, C.c_int, C.c_int64
_fp = C.c_void_p  # float* passed as raw addresses

# name -> (restype, argtypes); every symbol include/vitb200.h declares
SIGNATURES = {
    "vitb200_abi_version": (_i, []),
    "vitb200_last_error": (C.c_char_p, []),
    "vitb200_device_count": (_i, []),
    "vitb200_launch_count": (_i64, []),
    "vitb200_create": (_i, [C.POINTER(Config), _i, C.POINTER(_vp)]),
    "vitb200_destroy": (_i, [_vp]),
    "vitb200_num_params": (_i, [_vp]),
    "vitb200_param_info": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_i64)]),
    "vitb200_set_param": (_i, [_vp, C.c_char_p, _fp, C.POINTER(_i64), _i]),
    "vitb200_finalize_params": (_i, [_vp, _vp]),
    "vitb200_set_dropout_key": (_i, [_vp, C.c_uint64]),
    "vitb200_forward": (_i, [_vp, _vp, _fp, _i, _fp]),
    "vitb200_forward_host": (_i, [_vp, _vp, _fp, _i, _fp]),
    "vitb200_forward_attn": (_i, [_vp, _vp, _fp, _i, _fp, C.POINTER(C.c_int), _i, _fp]),
    "vitb200_submit_host": (_i, [_vp, _vp, _fp, _i, _fp]),
    "vitb200_wait_host": (_i, [_vp]),
    "vitb200_profile_forward": (_i, [_vp, _vp, _fp, _i, _fp, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "vitb200_debug_tokens": (_i, [_vp, _vp, _fp, _i]),
    "vitb200_train_forward": (_i, [_vp, _vp, _fp, _i, _fp]),
    "vitb200_backward": (_i, [_vp, _vp, _fp, _i]),
    "vitb200_backward_ex": (_i, [_vp, _vp, _fp, _i, _i, _fp]),
    "vitb200_get_grad": (_i, [_vp, _vp, C.c_char_p, _fp]),
    "vitb200_grads_buffer": (_i, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "vitb200_grad_device": (_i, [_vp, C.c_char_p, C.POINTER(C.c_void_p)]),
    "vitb200_set_leaf_flags": (_i, [_vp, C.POINTER(C.c_uint8)]),
    "vitb200_adamw_step": (_i, [_vp, _vp, C.POINTER(AdamW)]),
    "vitb200_optim_status": (_i, [_vp, _vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_float)]),
    "vitb200_optim_state": (_i, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "vitb200_get_param": (_i, [_vp, _vp, C.c_char_p, _fp]),
    "vitb200_softmax_xent": (_i, [_vp, _fp, _fp, _i, _i, C.c_float, C.c_float, _fp, _fp]),
    "vitb200_gemm_tc_wgrad": (_i, [_vp, _vp, _vp, _fp, _i, _i, _i, _i, _i]),
    "vitb200_attention_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i]),
    "vitb200_layernorm_bwd": (_i, [_vp, _vp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, C.c_float, _i]),
    "vitb200_gemm_tc": (_i, [_vp, _vp, _vp, _fp, _vp, _i, _i, _i, _i, _fp, _i, _i]),
    "vitb200_gemm_tc_dropout": (_i, [_vp, _vp, _vp, _fp, _vp, _i, _i, _i, _i, _fp, _i, _i, C.c_float, C.c_uint64, C.c_uint32]),
    "vitb200_gemm_tc_tokens": (_i, [_vp, _vp, _vp, _fp, _vp, _i, _i, _i, _i, _fp, _i, _fp, _i, C.c_float, C.c_uint64, C.c_uint32]),
    "vitb200_gemm_tc_ln": (_i, [_vp, _vp, _vp, _fp, _vp, _i, _i, _i, _i, _fp, _i, _fp, _i, _vp, _fp, _i, _fp, C.c_float]),
    "vitb200_gemm_tc_ln_slots": (_i, [_i, _i]),
    "vitb200_patch_embed_im2col": (_i, [_vp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _fp]),
    "vitb200_fold_layernorm": (_i, [_vp, _fp, _fp, _fp, _fp, _vp, _fp, _fp, _i, _i, _i, _i]),
    "vitb200_gemm_tc_e4m3": (_i, [_vp, _vp, _vp, _fp, _fp, _vp, _i, _i, _i, _i]),
    "vitb200_quantize_weight_e4m3": (_i, [_vp, _fp, _vp, _fp, _i, _i, _i]),
    "vitb200_gemm_f32": (_i, [_vp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _fp, _i]),
    "vitb200_layernorm": (_i, [_vp, _fp, _fp, _fp, _vp, _i, _i, _i]),
    "vitb200_attention_tc": (_i, [_vp, _vp, _vp, _i, _i, _i, _i]),
    "vitb200_attention_tc_lse": (_i, [_vp, _vp, _vp, _fp, _i, _i, _i, _i]),
    "vitb200_attention_probs": (_i, [_vp, _vp, _fp, _fp, _i, _i, _i, _i]),
    "vitb200_attention_f32": (_i, [_vp, _fp, _fp, _i, _i, _i]),
    "vitb200_patchify": (_i, [_vp, _fp, _vp, _i, _i, _i, _i, _i, _i, _i, _i]),
    "vitb200_patchify_tokens": (_i, [_vp, _fp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "vitb200_unpatchify": (_i, [_vp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "vitb200_cls_rows": (_i, [_vp, _fp, _fp, _fp, _i, _i, _i]),
    "vitb200_pool_layernorm": (_i, [_vp, _fp, _fp, _fp, _vp, _i, _i, _i, _i, _i]),
    "vitb200_pack_weight": (_i, [_vp, _fp, _vp, _i, _i, _i, _i]),
}

_lib = None


def load() -> C.CDLL:
    """Load the library once; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension is not built and vit_flax_b200 has no "
                "CPU fallback. Run `python -m vit_flax_b200.build` (needs nvcc) first.")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        got = lib.vitb200_abi_version()
        if got != ABI_VERSION:
            raise ImportError(f"libvitb200.so ABI version {got}, expected {ABI_VERSION}")
        _lib = lib
    return _lib


def check(rc: int) -> int:
    if rc < 0:
        msg = load().vitb200_last_error()
        raise VitB200Error(rc, msg.decode() if msg else "unknown error")
    return rc
