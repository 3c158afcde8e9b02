"""The checker of ``precision='fp8'``: the oracle's forward (``oracle.vit_torch``, LayerNorm-kernel schedule) with E4M3
rounding exactly where libvitb200 rounds to E4M3, and fp16 rounding where it keeps fp16 operands.

E4M3 sites: the two PreNorm LayerNorm outputs (no scale), the kernels of to_qkv, FeedForward Dense_0 and Dense_1 (one
fp32 scale per output column, ``amax / 448``), and the GELU output.  The three GEMMs compute ``(a8 @ w8) * scale + bias``
in fp32.  Everything else (patch embedding, attention, to_out, head) is the fp16 emulation of ``vit_torch``.  E4M3 is
torch ``float8_e4m3fn`` after clamping to +-448: round to nearest even with saturation, what
``cvt.rn.satfinite.e4m3x2.f32`` does.  It lives in tests/ so that oracle/ stays as it is."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import vit_torch

E4M3_MAX = 448.0
F16 = torch.float16


def e4m3(x):
    """fp32 -> nearest E4M3 value (ties to even, saturated), as fp32."""
    return torch.clamp(x, -E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(x.dtype)


def e4m3_codes(x):
    """fp32 tensor -> uint8 E4M3 codes (numpy), rounded as ``e4m3``."""
    return torch.clamp(torch.as_tensor(x, dtype=torch.float32), -E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn) \
        .view(torch.uint8).numpy()


def decode_e4m3(codes):
    """uint8 E4M3 codes -> float64 values (numpy)."""
    return torch.as_tensor(np.ascontiguousarray(codes, dtype=np.uint8)).view(torch.float8_e4m3fn).to(torch.float64).numpy()


def quantize_weight(W):
    """Flax kernel [K, N] fp32 -> (E4M3 values [K, N] as fp32, scale [N] fp32) with scale = amax_k |W| / 448 (1 for an
    all-zero column) and W8 = e4m3(W / scale): what ``vitb200_quantize_weight_e4m3`` computes."""
    W = torch.as_tensor(W, dtype=torch.float32)
    amax = W.abs().amax(dim=0)
    scale = torch.where(amax > 0, amax / torch.tensor(E4M3_MAX, dtype=torch.float32), torch.ones_like(amax))
    return e4m3(W / scale), scale


def _f16(x):
    return vit_torch._r(x, F16)


def _fp16_weight(W):
    return _f16(W), torch.ones(W.shape[1], dtype=W.dtype)


def _identity(x):
    return x


def _exact_weight(W):
    return W, torch.ones(W.shape[1], dtype=W.dtype)


def _ln(x, p, eps):
    return F.layer_norm(x, (x.shape[-1],), p["scale"], p["bias"], eps=eps)


def _fwd(p, images, *, patch_size, heads, dim, depth, pool, act, weight, r16, cls_token, ln_eps):
    ph, pw = (patch_size, patch_size) if not isinstance(patch_size, tuple) else patch_size
    x = torch.as_tensor(images).to(torch.float32)
    b, H, W, c = x.shape
    x = x.view(b, H // ph, ph, W // pw, pw, c).permute(0, 1, 3, 2, 4, 5).reshape(b, -1, ph * pw * c)
    x = r16(x) @ r16(p["Dense_0"]["kernel"]) + p["Dense_0"]["bias"]
    if cls_token:
        x = torch.cat([p["cls"].expand(b, -1, -1), x], dim=1)
    x = x + p["pos_embedding"][:, : x.shape[1]]
    tp = p["Transformer_0"]
    for l in range(depth):
        # Residual(PreNorm(Attention)): qkv = fp16((e4m3(LN(x)) @ W8) * s)
        a = tp[f"Attention_{l}"]
        w8, s = weight(a["Dense_0"]["kernel"])
        qkv = r16((act(_ln(x, tp[f"PreNorm_{2 * l}"]["LayerNorm_0"], ln_eps)) @ w8) * s)
        n = qkv.shape[1]
        q, k, v = (t.view(b, n, heads, vit_torch.DIM_HEAD).transpose(1, 2) for t in qkv.chunk(3, dim=-1))
        sc = (q @ k.transpose(-1, -2)) * vit_torch.DIM_HEAD ** -0.5
        e = torch.exp(sc - sc.amax(dim=-1, keepdim=True))
        o = r16(((r16(e) @ v) / e.sum(dim=-1, keepdim=True)).transpose(1, 2).reshape(b, n, heads * vit_torch.DIM_HEAD))
        if not (heads == 1 and vit_torch.DIM_HEAD == dim):
            o = F.linear(o, r16(a["Dense_1"]["kernel"]).t(), a["Dense_1"]["bias"])
        x = o + x
        # Residual(PreNorm(FeedForward)): h = e4m3(gelu((e4m3(LN(x)) @ W8) * s + b)), x += (h @ W8') * s' + b'
        f = tp[f"FeedForward_{l}"]
        w1, s1 = weight(f["Dense_0"]["kernel"])
        w2, s2 = weight(f["Dense_1"]["kernel"])
        h = act(F.gelu((act(_ln(x, tp[f"PreNorm_{2 * l + 1}"]["LayerNorm_0"], ln_eps)) @ w1) * s1 + f["Dense_0"]["bias"],
                       approximate="tanh"))
        x = (h @ w2) * s2 + f["Dense_1"]["bias"] + x
    x = x.mean(dim=1) if pool == "mean" else x[:, 0]
    x = _ln(x, p["LayerNorm_0"], ln_eps)
    return r16(x) @ r16(p["Dense_1"]["kernel"]) + p["Dense_1"]["bias"]


@torch.no_grad()
def vit_forward_fp8(variables, images, *, image_size=None, patch_size, num_classes=None, dim, depth, heads, mlp_dim=None,
                    pool="cls", rounding="e4m3", cls_token=True, ln_eps=1e-6):
    """Logits (numpy) of the ViT ``variables`` (Flax layout, ``{'params': ...}`` or the bare tree) on NHWC ``images``.

    ``rounding``: ``"e4m3"`` -- the fp8 precision; ``"fp16"`` -- every E4M3 site rounds to fp16 with unit weight scales
    instead, which is ``vit_torch.vit_forward(operand_dtype=float16)`` on the LayerNorm-kernel schedule; ``"none"`` --
    fp32 everywhere (the oracle itself).  ``cls_token`` / ``ln_eps`` cover SimpleViT's engine tree."""
    tree = variables["params"] if "params" in variables else variables
    p = vit_torch.tree_to_torch(tree)
    act, weight, r16 = {"e4m3": (e4m3, quantize_weight, _f16), "fp16": (_f16, _fp16_weight, _f16),
                        "none": (_identity, _exact_weight, _identity)}[rounding]
    return _fwd(p, images, patch_size=patch_size, heads=heads, dim=dim, depth=depth, pool=pool, act=act, weight=weight,
                r16=r16, cls_token=cls_token, ln_eps=ln_eps).numpy()
