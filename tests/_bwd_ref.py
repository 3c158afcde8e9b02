"""float64 references of the backward-pass kernels (csrc/backward.cu, csrc/attention_bwd_tc5.cu) and the error bounds
the GPU tests hold them to.  Plain torch on whatever device the inputs live on, so the GPU tests run them on CUDA next to
the kernel at full training sizes.

Two kinds of reference:
- SAME-ROUNDING: where the kernel rounds an intermediate to 16 bits, the reference rounds the exact value at the same
  place (``rnd``).  What is left between kernel and reference is fp32 arithmetic, the approximate exp2 / tanh of the
  SFU, and the final rounding, which the bounds below account for term by term.
- EXACT SUMS: the column-sum kernels are fed dyadic inputs (``dyadic``), so that every partial sum is exact in fp32
  whatever the order of the atomics, and their sums must equal the float64 sums bit for bit.
"""
from __future__ import annotations

import torch

U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}   # unit roundoff (half an ulp, relative) of the format
EPS32 = 2.0 ** -24                                              # unit roundoff of fp32
BT = 128                                                        # attention adjoint block edge (attention_bwd_tc5.cu)
# relative error of the adjoint kernel's P before it is rounded: the 64-term fp32 score, its log-sum-exp from the forward
# kernel (each <= 64 * 2^-24 * sum|q k| * 64^-0.5 * log2(e) ~ 1e-4 at |q|, |k| ~ 1.2 N(0, 1)) and ex2.approx (2^-22)
EPS_P = 2.0 ** -12


def rnd(x, tdt):
    """x rounded to the 16-bit type tdt (round to nearest even) and back; identity when tdt is None."""
    return x if tdt is None else x.to(tdt).to(x.dtype)


def dyadic(shape, bound, generator, device):
    """Random multiples of 2^-4 in [-bound, bound]: exact in fp16, bf16 and fp32, as are all their partial sums below
    2^24 * 2^-4 in magnitude."""
    k = int(bound * 16)
    return torch.randint(-k, k + 1, shape, generator=generator, device=device).to(torch.float32) / 16


def assert_sum_exact(n_terms, bound):
    """The premise of an exact-sum test: the largest possible |sum| stays below 2^24 units of 2^-4."""
    assert n_terms * bound * 16 < 2 ** 24, (n_terms, bound)


# ---------------------------------------------------------------- dropout masks (csrc/ptx.cuh: philox4x32_10 / dropout4)
def keep_mask(rows, cols, rate, site, key, device):
    """oracle/philox.keep_mask on the device (int64 arithmetic, products masked back to 32 bits)."""
    n = rows * cols
    M32 = 0xFFFFFFFF
    quad = torch.arange((n + 3) // 4, dtype=torch.int64, device=device)
    c0, c1 = quad & M32, quad >> 32
    c2 = torch.full_like(c0, site & M32)
    c3 = torch.zeros_like(c0)
    k0, k1 = key & M32, (key >> 32) & M32
    for _ in range(10):
        p0 = c0 * 0xD2511F53          # < 2^64: wraps in int64, the low 64 bits are the product's
        p1 = c2 * 0xCD9E8D57
        hi0, lo0 = (p0 >> 32) & M32, p0 & M32
        hi1, lo1 = (p1 >> 32) & M32, p1 & M32
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    words = torch.stack([c0, c1, c2, c3], dim=-1).reshape(-1)[:n]
    t = rate * 4294967296.0
    threshold = 0xFFFFFFFF if t >= 4294967295.0 else int(t)
    return (words >= threshold).view(rows, cols)


def inv_keep(rate):
    """1 / (1 - rate) as the kernels compute it, in fp32."""
    one = torch.tensor(1.0, dtype=torch.float32)
    return float(one / (one - torch.tensor(rate, dtype=torch.float32)))


def drop32(x32, rate, site, key):
    """The kernels' dropout of an fp32 [rows, cols] tensor: kept values times inv_keep in fp32, others 0."""
    if rate == 0.0:
        return x32
    keep = keep_mask(x32.shape[0], x32.shape[1], rate, site, key, x32.device)
    return torch.where(keep, x32 * inv_keep(rate), torch.zeros((), dtype=x32.dtype, device=x32.device))


# ---------------------------------------------------------------- attention adjoint
def attention_bwd(qkv16, o16, do16, heads, tdt, *, mutant=None):
    """Adjoint of softmax(Q K^T / 8) V per (image, head) rounded where attention_bwd_tc5.cu rounds (its header):

        P = exact softmax;  dV = round(P)^T dO;  dP = dO V^T;  D = rowsum(dO16 o O16)
        dS16 = round(P o (dP - D) / 8);  dQ = dS16 K;  dK = dS16^T Q;  outputs rounded to the format

    qkv16 [B, T, 3 * heads * 64], o16 / do16 [B, T, heads * 64] (16-bit or float; computed in float64).  tdt None: no
    rounding anywhere (then it is the exact adjoint).  Returns (dqkv [B, T, 3 * inner] float64, bound [same]) with

        |kernel - ref| <= 2u |ref| + (2u + EPS_P + T 2^-24) * mag

    where mag is the product of the magnitudes (|P|^T |dO| for dV; A |K|, A^T |Q| for dQ, dK with A = P o (|dO| |V|^T +
    |D|) / 8).  2u |ref| is the final rounding (kernel and reference may round to neighbours).  Each element of P16 or
    dS16 may be rounded to the other neighbour (one ulp = 2u of it) when the kernel's P differs from the exact one by
    EPS_P (above); dS also carries P's relative error unrounded; the fp32 tensor-core sums over T keys / queries add
    T 2^-24 of mag, the fp32 dP - D of 64 terms less than that.  All of it is bounded by the magnitude product mag.

    mutant (for the tests of the bound itself): 'dq_key_tile' drops key tile 1 from dQ (the streamed form's per-block
    dQ contribution), 'd_exact_o' takes D from the exact O instead of O16, 'lse_shift' normalises row i with row
    i + 1's log-sum-exp."""
    B, T, _ = qkv16.shape
    f = lambda t: t.to(torch.float64)
    x = f(qkv16).view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)          # [3, B, h, T, 64]
    q, k, v = x[0], x[1], x[2]
    do = f(do16).view(B, T, heads, 64).permute(0, 2, 1, 3)
    o = f(o16).view(B, T, heads, 64).permute(0, 2, 1, 3)
    s = q @ k.transpose(-1, -2) / 8.0
    lse = torch.logsumexp(s, dim=-1, keepdim=True)
    if mutant == "lse_shift":
        lse = torch.roll(lse, -1, dims=-2)
    p = torch.exp(s - lse)
    if mutant == "d_exact_o":
        o = p @ v
    u = U.get(tdt, 0.0)
    dv = rnd(p, tdt).transpose(-1, -2) @ do
    dp = do @ v.transpose(-1, -2)
    D = (do * o).sum(-1, keepdim=True)
    ds = rnd(p * (dp - D) / 8.0, tdt)
    ds_q = ds
    if mutant == "dq_key_tile":
        ds_q = ds.clone()
        ds_q[..., BT:2 * BT] = 0
    dq, dk = ds_q @ k, ds.transpose(-1, -2) @ q
    a = p * (do.abs() @ v.abs().transpose(-1, -2) + D.abs()) / 8.0
    mag_v = p.transpose(-1, -2) @ do.abs()
    mag_q, mag_k = a @ k.abs(), a.transpose(-1, -2) @ q.abs()
    c = 2 * u + EPS_P + T * EPS32
    pack = lambda t3: torch.stack(t3).permute(1, 3, 0, 2, 4).reshape(B, T, 3 * heads * 64)
    ref = [rnd(t, tdt) for t in (dq, dk, dv)]
    bound = [2 * u * r.abs() + c * m for r, m in zip(ref, (mag_q, mag_k, mag_v))]
    return pack(ref), pack(bound)


# ---------------------------------------------------------------- LayerNorm adjoint
def ln_stats(x, eps=1e-6):
    """mean, rstd, xhat of nn.LayerNorm() in float64 (flax: var = max(0, E[x^2] - E[x]^2))."""
    x = x.to(torch.float64)
    mean = x.mean(-1, keepdim=True)
    var = torch.clamp((x * x).mean(-1, keepdim=True) - mean * mean, min=0.0)
    rstd = torch.rsqrt(var + eps)
    return mean, rstd, (x - mean) * rstd


def ln_bwd(x, gamma, dy, eps=1e-6, x_err=0.0):
    """LayerNorm adjoint: -> (dx, dgamma, dbeta, bound_dx, bound_dgamma), float64.

    dx = rstd (g - a - xhat b), g = dy gamma, a = mean(g), b = mean(g xhat).  The kernel works in fp32 with rsqrtf
    (2 ulp); a row sum of dim terms carries at most k = 4 dim 2^-24 of the magnitudes it sums.  So xhat and rstd carry
    a relative error e = 2^-20 + k rstd mean|x| + 2 rstd x_err (x_err: absolute error of x itself, if it was computed),
    and
        |dx err| <= rstd (2^-20 |g - a - xhat b| + k (mean|g| + |xhat| mean|g xhat|)) + e (|dx| + rstd (|b| + |xhat| mean|g|))
        |dgamma err| <= sum_r (rows 2^-24 + e) |dy| (|xhat| + 1)      (fp32 sums of at most `rows` additions per path)"""
    dim = x.shape[-1]
    mean, rstd, xhat = ln_stats(x, eps)
    x64, dy64 = x.to(torch.float64), dy.to(torch.float64)
    g = dy64 * gamma.to(torch.float64)
    a = g.mean(-1, keepdim=True)
    b = (g * xhat).mean(-1, keepdim=True)
    dx = rstd * (g - a - xhat * b)
    k = 4 * dim * EPS32
    e = 2.0 ** -20 + k * rstd * x64.abs().mean(-1, keepdim=True) + 2 * rstd * x_err
    gm = g.abs().mean(-1, keepdim=True)
    bound_dx = (rstd * (2.0 ** -20 * (g - a - xhat * b).abs() + k * (gm + xhat.abs() * (g * xhat).abs().mean(-1, keepdim=True)))
                + e * (dx.abs() + rstd * (b.abs() + xhat.abs() * gm)))
    rows = x.shape[0]
    bound_dg = ((rows * EPS32 + e) * dy64.abs() * (xhat.abs() + 1)).sum(0)
    return dx, (dy64 * xhat).sum(0), dy64.sum(0), bound_dx, bound_dg


def colsum_bound(v, rows_per_path):
    """fp32 column sums of v [rows, cols] whose partial sums pass through at most rows_per_path additions:
    |err| <= rows_per_path 2^-24 sum_r |v|."""
    return rows_per_path * EPS32 * v.to(torch.float64).abs().sum(0)


# ---------------------------------------------------------------- GELU (tanh form, vit.py:49)
K0, K1 = 0.7978845608028654, 0.044715


def gelu_tanh(x):
    x = x.to(torch.float64)
    return 0.5 * x * (1 + torch.tanh(K0 * x * (1 + K1 * x * x)))


def gelu_tanh_grad(x):
    """d/dx of gelu_tanh, and its error bound when tanh is tanh.approx (2^-11 relative) and the rest fp32."""
    x = x.to(torch.float64)
    t = torch.tanh(K0 * x * (1 + K1 * x * x))
    grad = 0.5 * (1 + t) + 0.5 * x * (1 - t * t) * K0 * (1 + 3 * K1 * x * x)
    dgrad_dt = (0.5 - x * t * K0 * (1 + 3 * K1 * x * x)).abs()
    bound = dgrad_dt * 2.0 ** -11 * t.abs() + 2.0 ** -20 * (1 + x.abs())
    return grad, bound


# ---------------------------------------------------------------- head: pool + LayerNorm, Dense
def pool_ln_bwd(x, dy, gamma, pool_mean, eps=1e-6):
    """Adjoint of LayerNorm(pool(x)): x [B, T, D], dy [B, D] -> (dpooled_row [B, D], dx [B, T, D], dgamma, dbeta,
    bound_row [B, D]); dpooled_row is the gradient of one token row (mean: the pooled gradient / T).  The pooled
    vector of the mean pool is an fp32 sum over T (relative error T 2^-24 of mean|x|), added to the LayerNorm bound."""
    B, T, D = x.shape
    x64 = x.to(torch.float64)
    pooled = x64.mean(1) if pool_mean else x64[:, 0]
    x_err = 2 * T * EPS32 * x64.abs().mean(1).amax(-1, keepdim=True) if pool_mean else 0.0
    dp, dg, db, bnd, _ = ln_bwd(pooled, gamma, dy, eps, x_err)
    if pool_mean:
        dp, bnd = dp / T, bnd / T
        dx = dp.unsqueeze(1).expand(B, T, D)
    else:
        dx = torch.zeros((B, T, D), dtype=torch.float64, device=x.device)
        dx[:, 0] = dp
    return dp, dx, dg, db, bnd


def head_bwd(pooled, dl, W):
    """Head Dense adjoint (fp32 kernels): -> (dpooled, dW, dbias, bound_dpooled, bound_dW)."""
    p, d, w = (t.to(torch.float64) for t in (pooled, dl, W))
    return (d @ w.t(), p.t() @ d, d.sum(0),
            W.shape[1] * EPS32 * (d.abs() @ w.abs().t()), pooled.shape[0] * EPS32 * (p.abs().t() @ d.abs()))


def token_grads(dx, cls_slot):
    """vit.py:151-153 adjoint: dx [B, T, D] -> (dpos [T, D], dcls [D] or None, dbias [D])."""
    dpos = dx.to(torch.float64).sum(0)
    if cls_slot:
        return dpos, dpos[0], dpos[1:].sum(0)
    return dpos, None, dpos.sum(0)


# ---------------------------------------------------------------- every leaf, float64 on the device
def vjp_on_device(variables, images, dlogits, *, chunk=16, device="cuda", **cfg):
    """oracle.vit_torch._vit_forward under float64 autograd on `device`, in chunks of `chunk` images.  The parameter
    gradients of the chunks are summed (the map is linear over the batch, so this is the batch's gradient); the image
    gradients are concatenated.  Dropout 0 only (oracle._drop builds its masks on the CPU).
    -> (logits [B, classes], grads as a tree like variables['params'], dimages like images), numpy float64."""
    from oracle import vit_torch
    assert not cfg.get("dropout") and not cfg.get("emb_dropout")
    tree = variables["params"] if "params" in variables else variables

    def conv(t):
        if isinstance(t, dict) or hasattr(t, "items"):
            return {k: conv(v) for k, v in t.items()}
        return torch.as_tensor(t).to(device, torch.float64).clone().requires_grad_(True)

    p = conv(tree)
    imgs = torch.as_tensor(images)
    dls = torch.as_tensor(dlogits)
    logits, dimg = [], []
    for b0 in range(0, imgs.shape[0], chunk):
        x = imgs[b0:b0 + chunk].to(device, torch.float64).requires_grad_(True)
        with torch.enable_grad():
            out = vit_torch._vit_forward({"params": p}, x, **cfg)
            (out * dls[b0:b0 + chunk].to(device, torch.float64)).sum().backward()   # .grad accumulates over chunks
        logits.append(out.detach().cpu())
        dimg.append(x.grad.detach().cpu())

    def grads(t):
        if isinstance(t, dict):
            return {k: grads(v) for k, v in t.items()}
        return (t.grad if t.grad is not None else torch.zeros_like(t)).detach().cpu().numpy()

    return torch.cat(logits).numpy(), grads(p), torch.cat(dimg).numpy()
