"""The checker of attention maps: the forward of ``oracle.vit_numpy`` / ``oracle.simple_vit_numpy`` with the attention
weights ``softmax(q k^T * 64^-0.5)`` of every layer kept (vit.py:73-75, simple_vit.py:67-68), in float64.

``rounding='fp16' | 'bf16' | 'e4m3'`` emulates where the tensor-core path rounds the INPUTS of those weights: the PreNorm
LayerNorm output and the to_qkv kernel (the GEMM operands) and q / k (the GEMM's 16-bit output); the residual stream and
the softmax stay float64.  Its distance to the exact maps on the same inputs is the error floor of the format there, and
the GPU maps are held to a multiple of it -- the method of tests/_fp8_oracle.py.  It lives in tests/ so that oracle/ stays
as it is."""
import numpy as np
import torch

from oracle import simple_vit_numpy as svn
from oracle import vit_numpy as vn
from oracle.vit_numpy import DIM_HEAD, _drop, dense, layer_norm, pair, patchify, softmax_last

_FMT = {"fp16": torch.float16, "bf16": torch.bfloat16}

# GPU maps against the float64 oracle: |P - P_ref| <= FLOOR_MULT * (the emulation's error floor on the same inputs) +
# FLOOR_ABS.  The multiple covers what the emulation leaves out -- the 16-bit rounding of the residual stream by the
# earlier layers (to_out / FeedForward operands), and the LayerNorm fold, which rounds x and diag(gamma) W instead of
# LayerNorm(x) and W -- each of the same order as the rounding emulated.
FLOOR_MULT = 4.0
FLOOR_ABS = 1e-6


def round16(x, fmt):
    """``x`` rounded to the 16-bit format ``fmt`` (nearest even) and back to float64; ``fmt`` None: ``x`` itself."""
    if fmt is None:
        return x
    return torch.as_tensor(np.asarray(x, np.float64)).to(_FMT[fmt]).to(torch.float64).numpy()


def _qkv(xn, W, fmt):
    """to_qkv (vit.py:68) with the operands rounded as the GPU rounds them.  ``'e4m3'`` is the fp8 precision: E4M3
    LayerNorm output, E4M3 weights with one scale per column (tests/_fp8_oracle.py), fp16 q / k / v."""
    if fmt == "e4m3":
        from _fp8_oracle import e4m3, quantize_weight
        w8, scale = quantize_weight(W)
        a8 = e4m3(torch.as_tensor(xn, dtype=torch.float32)).to(torch.float64)
        return round16(((a8 @ w8.to(torch.float64)) * scale.to(torch.float64)).numpy(), "fp16")
    return round16(round16(xn, fmt) @ round16(W, fmt), fmt)


def _maps(xn, p_qkv, heads, fmt):
    """Attention weights [b, heads, n, n] of the to_qkv Dense ``p_qkv`` (no bias, vit.py:68) on the normalised tokens
    ``xn`` [b, n, dim]."""
    b, n, _ = xn.shape
    qkv = _qkv(xn, np.asarray(p_qkv["kernel"], np.float64), fmt)
    q, k, _ = np.split(qkv, 3, axis=-1)                                        # vit.py:69

    def th(t):                                                                 # vit.py:71
        return t.reshape(b, n, heads, DIM_HEAD).transpose(0, 2, 1, 3)

    return softmax_last(np.einsum("bhid,bhjd->bhij", th(q), th(k)) * DIM_HEAD ** -0.5)   # vit.py:73-75


def _stack(maps, layers):
    return np.stack([maps[l] for l in layers], axis=1)


def vit_attention_maps(variables, images, *, layers=None, rounding=None, image_size, patch_size, num_classes, dim,
                       depth, heads, mlp_dim, pool="cls", dropout=0.0, emb_dropout=0.0, dropout_key=None):
    """``(logits [B, classes], maps [B, len(layers), heads, T, T])`` of ``ViT`` (vit.py:127-167) in float64; ``layers``
    default every layer.  Dropout as ``vit_numpy.vit_forward`` applies it (the Philox masks of libvitb200); no site
    touches the attention weights."""
    p = variables["params"] if "params" in variables else variables
    layers = list(range(depth)) if layers is None else list(layers)
    ph, pw = pair(patch_size)
    x = dense(patchify(np.asarray(images, np.float64), ph, pw), p["Dense_0"])   # vit.py:146-147
    b, n, _ = x.shape
    cls = np.broadcast_to(np.asarray(p["cls"], np.float64), (b, 1, dim))
    x = np.concatenate([cls, x], axis=1) + np.asarray(p["pos_embedding"], np.float64)[:, : n + 1]   # vit.py:151-153
    x = _drop(x, (emb_dropout, dropout_key), 0)                                 # vit.py:155
    drop = (dropout, dropout_key) if dropout else None
    tp = p["Transformer_0"]
    maps = {}
    for l in range(depth):                                                      # vit.py:108-110 (vit_numpy.transformer)
        xn = layer_norm(x, tp[f"PreNorm_{2 * l}"]["LayerNorm_0"])
        if l in layers:
            maps[l] = _maps(xn, tp[f"Attention_{l}"]["Dense_0"], heads, rounding)
        x = vn.attention(xn, tp[f"Attention_{l}"], heads, dim, drop, 1 + 3 * l) + x
        x = vn.feed_forward(layer_norm(x, tp[f"PreNorm_{2 * l + 1}"]["LayerNorm_0"]), tp[f"FeedForward_{l}"], drop,
                            2 + 3 * l) + x
    x = x.mean(axis=1) if pool == "mean" else x[:, 0]                           # vit.py:159
    logits = dense(layer_norm(x, p["LayerNorm_0"]), p["Dense_1"])              # vit.py:163-165
    return logits, _stack(maps, layers)


def simple_vit_attention_maps(variables, img, *, layers=None, rounding=None, image_size, patch_size, num_classes, dim,
                              depth, heads, mlp_dim, channels=3):
    """``SimpleViT`` (simple_vit.py:110-134, ``img`` NCHW): ``(logits, maps)`` as ``vit_attention_maps``, T = num_patches."""
    p = variables["params"] if "params" in variables else variables
    layers = list(range(depth)) if layers is None else list(layers)
    ph, pw = pair(patch_size)
    x = np.asarray(img, np.float64)
    b, c, H, W = x.shape
    gh, gw = H // ph, W // pw
    x = x.reshape(b, c, gh, ph, gw, pw).transpose(0, 2, 4, 3, 5, 1).reshape(b, gh * gw, ph * pw * c)   # simple_vit.py:125
    if "Sequential_0" in p:
        patch, head_norm, head_dense = p["Dense_0"], p["Sequential_0"]["layers_0"], p["Sequential_0"]["layers_1"]
    else:
        patch, head_norm, head_dense = p["Dense_1"], p["LayerNorm_0"], p["Dense_0"]
    x = dense(x, patch) + svn.posemb_sincos_2d(gh, gw, dim)                     # simple_vit.py:126-128
    tp = p["Transformer_0"]
    maps = {}
    for l in range(depth):                                                      # simple_vit.py:92-95
        a = tp[f"Attention_{l}"]
        if l in layers:
            maps[l] = _maps(svn.layer_norm_nobias(x, a["LayerNorm_0"]), a["Dense_0"], heads, rounding)
        x = svn.attention(x, a, heads) + x
        x = svn.feed_forward(x, tp[f"FeedForward_{l}"]) + x
    logits = dense(svn.layer_norm_nobias(x.mean(axis=1), head_norm), head_dense)   # simple_vit.py:117-120,131-134
    return logits, _stack(maps, layers)


def error_floor(maps_emulated, maps_exact):
    """The largest |difference| between the emulated and the exact maps: the format's floor at these inputs."""
    return float(np.abs(maps_emulated - maps_exact).max())


def tolerance(floor):
    return FLOOR_MULT * floor + FLOOR_ABS
