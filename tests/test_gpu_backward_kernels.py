"""The backward pass kernel by kernel at training sizes, on a real B200, against the float64 references of
tests/_bwd_ref.py (run on the GPU next to the kernels).

- The attention adjoint (attention_bwd_tc5.cu) is held to a same-rounding reference on EVERY (image, head) of
  ViT-B/16, ViT-L/16, ViT-H/14 and 512-px batches, plus repeated launches and batch-neighbour independence: the
  scheduling of thousands of units over 148 persistent CTAs is what these catch.
- The non-GEMM kernels of backward.cu run through their per-kernel entry points at the shapes where they go wrong:
  template boundaries of the LayerNorm adjoint, rows past its persistent grid, ragged columns of the row passes.
  Every column sum is fed dyadic inputs and must equal the float64 sum bit for bit (one dropped or doubled row of 50k
  would show); the rest meet a stated fp32 bound (tests/_bwd_ref.py).
- Every leaf and the image gradient of the full ViT-B/16 at batch 256 against float64 autograd on the device."""
import ctypes as C
import math
import time

import numpy as np
import pytest
import torch

import _bwd_ref as R
from vit_flax_b200 import _lib, init_params, perturb_params
from vit_flax_b200.engine import Engine
from vit_flax_b200.params import flatten_params
from vit_flax_b200.runtime import clear_cache
from _util import C2, images_for

pytestmark = pytest.mark.gpu

DT16 = {"fp16": (_lib.DT_F16, torch.float16), "bf16": (_lib.DT_BF16, torch.bfloat16)}
KEY, SITE = 0x0DDBA11CAFEF00D5, 11
SMS = 148


@pytest.fixture(scope="module")
def lib(lib_built):
    assert lib_built.vitb200_device_count() >= 1, "no sm_100 device"
    return lib_built


@pytest.fixture(autouse=True)
def _free():
    yield
    clear_cache()
    torch.cuda.empty_cache()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def within(got, want, bound):
    """max of |got - want| / bound (<= 1 passes); NaN anywhere in got fails."""
    got = got.double()
    assert torch.isfinite(got).all(), "non-finite output (an element never written?)"
    return float(((got - want).abs() / bound.clamp_min(1e-300)).max())


# ================================================================ A. attention adjoint
def _attn_launch(lib, qkv, o, do, B, T, heads, dt, tdt):
    dqkv = torch.full((B * T, 3 * heads * 64), float("nan"), dtype=tdt, device="cuda")
    _lib.check(lib.vitb200_attention_bwd(stream(), qkv.data_ptr(), o.data_ptr(), do.data_ptr(), dqkv.data_ptr(), B, T, heads, dt))
    torch.cuda.synchronize()
    return dqkv


def _attn_ratio(qkv, o, do, dqkv, B, T, heads, tdt, cols=slice(None)):
    """worst |kernel - ref| / bound over every (image, head), the reference in float64 on the GPU in chunks of images"""
    chunk = max(1, min(B, int(1e8 // (heads * T * T))))
    worst = 0.0
    for b0 in range(0, B, chunk):
        nb = min(chunk, B - b0)
        rows = slice(b0 * T, (b0 + nb) * T)
        ref, bound = R.attention_bwd(qkv[rows].view(nb, T, -1), o[rows].view(nb, T, -1), do[rows].view(nb, T, -1), heads, tdt)
        worst = max(worst, within(dqkv[rows].view(nb, T, -1)[..., cols], ref[..., cols], bound[..., cols]))
    return worst


ATTN_SHAPES = [(256, 197, 12), (128, 197, 16), (64, 257, 16), (16, 1025, 16),    # ViT-B/16, L/16, H/14, 512 px
               (5, 1, 2), (5, 16, 2), (4, 129, 2), (3, 255, 2), (3, 256, 2), (2, 385, 2),   # tile edges
               (8, 197, 6), (8, 257, 6), (8, 197, 10), (8, 257, 10)]              # heads * 8 not a multiple of 32


@pytest.mark.parametrize("B,T,heads", ATTN_SHAPES)
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_attention_bwd_every_unit(lib, B, T, heads, fmt):
    """dqkv of vitb200_attention_bwd on every (image, head) against the same-rounding reference, bound derived in
    _bwd_ref.attention_bwd (2u |ref| + (2u + 2^-12 + T 2^-24) * magnitude product).  dqkv starts as NaN.  Three launches
    back to back: the resident form (T <= 208) gives the same bits each time; the streamed form the same dK / dV bits,
    its dQ (fp32 red.add, order-dependent) within the bound each time.  At the training sizes a few images are also run
    alone at batch 1 and must give the bits they had inside the full batch (dK / dV only when streamed)."""
    dt, tdt = DT16[fmt]
    inner = heads * 64
    g = gen(B * T + heads)
    qkv = (torch.randn((B * T, 3 * inner), device="cuda", generator=g) * 1.2).to(tdt)
    do = torch.randn((B * T, inner), device="cuda", generator=g).to(tdt)
    o = torch.empty((B * T, inner), dtype=tdt, device="cuda")          # the forward's output, as train_forward keeps it
    _lib.check(lib.vitb200_attention_tc(stream(), qkv.data_ptr(), o.data_ptr(), B, T, heads, dt))
    streamed = T > 208
    kv = slice(inner, 3 * inner)
    runs = [_attn_launch(lib, qkv, o, do, B, T, heads, dt, tdt) for _ in range(3)]
    worst = _attn_ratio(qkv, o, do, runs[0], B, T, heads, tdt)
    assert worst <= 1.0, worst
    for r in runs[1:]:
        if streamed:
            assert torch.equal(r[:, kv], runs[0][:, kv])
            assert _attn_ratio(qkv, o, do, r, B, T, heads, tdt, cols=slice(0, inner)) <= 1.0
        else:
            assert torch.equal(r, runs[0])
    if B >= 16:
        for b in (0, B // 2 + 1, B - 1):
            rows = slice(b * T, (b + 1) * T)
            alone = _attn_launch(lib, qkv[rows].contiguous(), o[rows].contiguous(), do[rows].contiguous(), 1, T, heads, dt, tdt)
            cols = kv if streamed else slice(None)
            assert torch.equal(alone[:, cols], runs[0][rows, cols]), b


# ================================================================ B. backward.cu, per kernel
def _ln_paths(rows):
    """longest chain of fp32 additions behind one column sum of ln_bwd_kernel: rows of a warp, 4 warps, the blocks' atomics"""
    grid = min((rows + 3) // 4, 3 * SMS)
    return math.ceil(rows / (4 * grid)) + 4 + grid


def _ln_case(lib, rows, dim, fmt, accumulate, rate):
    dt, tdt = DT16[fmt]
    g = gen(rows * 7 + dim + accumulate)
    x = torch.randn((rows, dim), device="cuda", generator=g) * 2 + 0.5
    gamma = torch.randn(dim, device="cuda", generator=g) * 0.5 + 1
    dy = R.dyadic((rows, dim), 4, g, "cuda").to(tdt)
    R.assert_sum_exact(rows, 4)
    dx0 = torch.randn((rows, dim), device="cuda", generator=g)
    dx = dx0.clone() if accumulate else torch.full((rows, dim), float("nan"), device="cuda")
    dgamma, dbeta, dbn = (torch.zeros(dim, device="cuda") for _ in range(3))
    dx16 = torch.full((rows, dim), float("nan"), dtype=tdt, device="cuda")
    _lib.check(lib.vitb200_layernorm_bwd_ex(stream(), dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), dx.data_ptr(),
                                            dgamma.data_ptr(), dbeta.data_ptr(), rows, dim, dt, 1e-6, accumulate,
                                            dx16.data_ptr(), dbn.data_ptr(), rate, KEY, SITE))
    torch.cuda.synchronize()
    rdx, rdg, rdb, bdx, bdg = R.ln_bwd(x, gamma, dy)
    if accumulate:
        rdx = rdx + dx0.double()
        bdx = bdx + R.EPS32 * rdx.abs()
    assert within(dx, rdx, bdx) <= 1.0
    assert within(dgamma, rdg, bdg) <= 1.0
    assert torch.equal(dbeta.double(), rdb), "dbeta of dyadic dy must be the exact sum"
    masked = R.drop32(dx, rate, SITE, KEY)                  # dx is stored unmasked; dx16 and dbias_next are masked
    assert torch.equal(dx16, masked.to(tdt)), "dx16 must be the kernel's dx, masked in fp32, rounded once"
    assert within(dbn, masked.double().sum(0), R.colsum_bound(masked, _ln_paths(rows))) <= 1.0


LN_DIMS = [64, 72, 200, 256, 260, 768, 772, 1024, 1028, 1280]     # each KV template's edge and just past it


@pytest.mark.parametrize("dim", LN_DIMS)
@pytest.mark.parametrize("rows", [1, 3, 4 * 3 * SMS + 5])         # past the persistent grid's stride: prefetch off the end
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_layernorm_bwd_fused_outputs(lib, rows, dim, fmt):
    for accumulate in (0, 1):
        for rate in (0.0, 0.5, 0.1):
            _ln_case(lib, rows, dim, fmt, accumulate, rate)


@pytest.mark.parametrize("dim", [768, 1280])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_layernorm_bwd_fused_outputs_vit_b16_batch_256(lib, dim, fmt):
    for accumulate, rate in ((1, 0.5), (0, 0.1), (1, 0.0)):
        _ln_case(lib, 256 * 197, dim, fmt, accumulate, rate)


def _rowpass_paths(rows, cols):
    """longest chain of fp32 additions behind one column sum of rowpass_colsum_kernel (rowpass_grid in backward.cu)"""
    gx = (cols + 255) // 256
    gy = max(1, min((rows + 7) // 8, max(1, 4 * SMS // gx)))
    return math.ceil(rows / (8 * gy)) + 8 + gy


ROWPASS = [(1, 8), (7, 264), (1000, 768), (50432, 768), (50432, 3072), (3000, 5120), (50432, 5120)]


@pytest.mark.parametrize("rows,cols", ROWPASS)
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_cast16_colsum_exact(lib, rows, cols, fmt):
    """Mode 0: y16 = round(Dropout(x)) and sums += column sums of the masked fp32 values -- bit for bit on dyadic x."""
    dt, tdt = DT16[fmt]
    g = gen(rows + cols)
    x = R.dyadic((rows, cols), 4, g, "cuda")
    for rate in (0.0, 0.5):
        R.assert_sum_exact(rows, 4 * R.inv_keep(rate))
        y = torch.full((rows, cols), float("nan"), dtype=tdt, device="cuda")
        sums = torch.full((cols,), 0.5, device="cuda")                   # accumulates
        _lib.check(lib.vitb200_cast16_colsum(stream(), x.data_ptr(), y.data_ptr(), sums.data_ptr(), rows, cols, dt, rate, KEY, SITE))
        torch.cuda.synchronize()
        masked = R.drop32(x, rate, SITE, KEY)
        assert torch.equal(y, masked.to(tdt))
        assert torch.equal(sums.double(), masked.double().sum(0) + 0.5), rate


@pytest.mark.parametrize("rows,cols", ROWPASS)
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_gelu_bwd_colsum(lib, rows, cols, fmt):
    """Mode 1: dpre16 = round(Dropout(dhid * gelu'(pre))) against the float64 derivative within the tanh.approx bound
    (_bwd_ref.gelu_tanh_grad) plus one rounding; the sums are of the ROUNDED outputs (what the GEMMs see), held to the
    fp32 summation bound of the kernel's addition chains.  Also in place (dpre = dhid), as the backward runs it."""
    dt, tdt = DT16[fmt]
    u = R.U[tdt]
    g = gen(rows * 3 + cols)
    pre = (torch.randn((rows, cols), device="cuda", generator=g) * 2).to(tdt)
    dhid = torch.randn((rows, cols), device="cuda", generator=g).to(tdt)
    grad, gbound = R.gelu_tanh_grad(pre)
    for rate, in_place in ((0.0, False), (0.5, True)):
        out = dhid.clone() if in_place else torch.full((rows, cols), float("nan"), dtype=tdt, device="cuda")
        sums = torch.zeros(cols, device="cuda")
        _lib.check(lib.vitb200_gelu_bwd_colsum(stream(), pre.data_ptr(), out.data_ptr() if in_place else dhid.data_ptr(),
                                               out.data_ptr(), sums.data_ptr(), rows, cols, dt, rate, KEY, SITE))
        torch.cuda.synchronize()
        scale = torch.ones_like(grad) if rate == 0 else R.keep_mask(rows, cols, rate, SITE, KEY, "cuda").double() * R.inv_keep(rate)
        want = dhid.double() * grad * scale
        bound = u * want.abs() + dhid.double().abs() * gbound * scale + 2.0 ** -24
        assert within(out, want, bound) <= 1.0
        assert within(sums, out.double().sum(0), R.colsum_bound(out, _rowpass_paths(rows, cols))) <= 1.0


@pytest.mark.parametrize("n", [8, 264 * 7, 50432 * 3072])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_gelu_fwd(lib, n, fmt):
    """hid16 = round(Dropout(gelu_tanh(pre16))): tanh.approx moves gelu by 0.5 |x| 2^-11 |t|, plus one rounding."""
    dt, tdt = DT16[fmt]
    pre = (torch.randn(n, device="cuda", generator=gen(n)) * 2).to(tdt)
    x = pre.double()
    t = torch.tanh(R.K0 * x * (1 + R.K1 * x * x))
    for rate in (0.0, 0.1):
        hid = torch.full((n,), float("nan"), dtype=tdt, device="cuda")
        _lib.check(lib.vitb200_gelu_fwd(stream(), pre.data_ptr(), hid.data_ptr(), n, dt, rate, KEY, SITE))
        torch.cuda.synchronize()
        scale = 1.0 if rate == 0 else R.keep_mask(1, n, rate, SITE, KEY, "cuda").view(n).double() * R.inv_keep(rate)
        want = R.gelu_tanh(pre) * scale
        bound = R.U[tdt] * want.abs() + (0.5 * x.abs() * 2.0 ** -11 * t.abs() + 2.0 ** -20 * (1 + x.abs())) * scale + 2.0 ** -24
        assert within(hid, want, bound) <= 1.0


def test_dropout_inplace(lib):
    n = 50432 * 768
    x0 = torch.randn(n, device="cuda", generator=gen(5))
    for rate in (0.0, 0.5, 0.1):
        x = x0.clone()
        _lib.check(lib.vitb200_dropout_inplace(stream(), x.data_ptr(), n, rate, KEY, SITE))
        torch.cuda.synchronize()
        assert torch.equal(x, R.drop32(x0.view(1, n), rate, SITE, KEY).view(n)), rate


@pytest.mark.parametrize("pool", [0, 1])
@pytest.mark.parametrize("T", [1, 17, 197, 1025])
@pytest.mark.parametrize("dim", [64, 200, 768, 1280])
@pytest.mark.parametrize("batch", [1, 256])
def test_pool_layernorm_bwd(lib, pool, T, dim, batch):
    """Adjoint of LayerNorm(pool(x)): dpooled within the LayerNorm bound, dx (prefilled NaN) written on every row --
    the pooled gradient on row 0 and zeros elsewhere (cls), the same row everywhere (mean) -- and dbeta exact."""
    g = gen(pool + T + dim + batch)
    x = torch.randn((batch, T, dim), device="cuda", generator=g) * 1.5 + 0.3
    gamma = torch.randn(dim, device="cuda", generator=g) * 0.5 + 1
    dy = R.dyadic((batch, dim), 4, g, "cuda")
    dpooled = torch.full((batch, dim), float("nan"), device="cuda")
    dx = torch.full((batch, T, dim), float("nan"), device="cuda")
    dgamma, dbeta = torch.zeros(dim, device="cuda"), torch.zeros(dim, device="cuda")
    _lib.check(lib.vitb200_pool_layernorm_bwd(stream(), x.data_ptr(), dy.data_ptr(), gamma.data_ptr(), dpooled.data_ptr(),
                                              dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), batch, T, dim, pool, 1e-6))
    torch.cuda.synchronize()
    rdp, _, rdg, rdb, bnd = R.pool_ln_bwd(x, dy, gamma, pool)
    assert within(dpooled, rdp, bnd) <= 1.0
    _, _, _, _, bdg = R.ln_bwd(x.mean(1) if pool else x[:, 0], gamma, dy)
    assert within(dgamma, rdg, bdg * (2 if pool else 1)) <= 1.0
    assert torch.equal(dbeta.double(), rdb)
    assert torch.equal(dx[:, 0], dpooled)
    if pool:
        assert torch.equal(dx, dpooled.unsqueeze(1).expand(batch, T, dim))
    else:
        assert torch.count_nonzero(dx[:, 1:]) == 0 and not dx.isnan().any()


@pytest.mark.parametrize("batch,dim,classes", [(256, 768, 1000), (3, 64, 7), (256, 1280, 1001), (1, 192, 1), (256, 1024, 1)])
def test_head_bwd(lib, batch, dim, classes):
    """Head Dense adjoint (fp32): dpooled and dW within fp32 dot-product bounds, the bias gradient exact (dyadic
    cotangent), and dpooled the same bits with dW / dbias skipped (the image-only backward)."""
    g = gen(batch + dim + classes)
    pooled = torch.randn((batch, dim), device="cuda", generator=g)
    dl = R.dyadic((batch, classes), 4, g, "cuda")
    R.assert_sum_exact(batch, 4)
    W = torch.randn((dim, classes), device="cuda", generator=g) / math.sqrt(dim)
    dW0 = torch.randn((dim, classes), device="cuda", generator=g)
    dW, dbias = dW0.clone(), torch.full((classes,), 0.25, device="cuda")
    dpooled = torch.full((batch, dim), float("nan"), device="cuda")
    _lib.check(lib.vitb200_head_bwd(stream(), pooled.data_ptr(), dl.data_ptr(), W.data_ptr(), dW.data_ptr(), dbias.data_ptr(),
                                    dpooled.data_ptr(), batch, dim, classes))
    torch.cuda.synchronize()
    rdp, rdW, rdb, bdp, bdW = R.head_bwd(pooled, dl, W)
    assert within(dpooled, rdp, bdp + 1e-30) <= 1.0
    assert within(dW, rdW + dW0.double(), bdW + R.EPS32 * (rdW + dW0.double()).abs()) <= 1.0
    assert torch.equal(dbias.double(), rdb + 0.25)
    dp2 = torch.full((batch, dim), float("nan"), device="cuda")
    _lib.check(lib.vitb200_head_bwd(stream(), None, dl.data_ptr(), W.data_ptr(), None, None, dp2.data_ptr(), batch, dim, classes))
    torch.cuda.synchronize()
    assert torch.equal(dp2, dpooled)


@pytest.mark.parametrize("cls_slot", [0, 1])
@pytest.mark.parametrize("T", [1, 17, 197, 1025])
@pytest.mark.parametrize("batch,dim", [(1, 768), (256, 768), (7, 200)])
def test_token_grads_exact(lib, cls_slot, T, batch, dim):
    """dpos = sum over the batch, dcls = dpos[0], patch-bias gradient = sum of the other rows (all of them without a
    class token) -- bit for bit on dyadic dx (|x| <= 2 keeps 256 x 1025 rows below 2^24 units)."""
    g = gen(cls_slot + T + batch + dim)
    dx = R.dyadic((batch, T, dim), 2, g, "cuda")
    R.assert_sum_exact(batch * T, 2)
    dpos = torch.zeros((T, dim), device="cuda")
    dcls, dbias = torch.full((dim,), 0.5, device="cuda"), torch.full((dim,), 0.25, device="cuda")
    _lib.check(lib.vitb200_token_grads(stream(), dx.data_ptr(), dpos.data_ptr(), dcls.data_ptr(), dbias.data_ptr(),
                                       batch, T, dim, cls_slot))
    torch.cuda.synchronize()
    rpos, rcls, rbias = R.token_grads(dx, cls_slot)
    assert torch.equal(dpos.double(), rpos)
    assert torch.equal(dbias.double(), rbias + 0.25)
    assert torch.equal(dcls.double(), (rcls + 0.5) if cls_slot else torch.full_like(rbias, 0.5))


def test_entry_points_check_their_arguments(lib):
    a = torch.zeros(64, device="cuda")
    rc = lib.vitb200_layernorm_bwd_ex(stream(), a.data_ptr(), a.data_ptr(), a.data_ptr(), a.data_ptr(), a.data_ptr(),
                                      a.data_ptr(), 1, 64, _lib.DT_F16, 1e-6, 0, None, a.data_ptr(), 0.0, 0, 0)
    assert rc == -1 and b"dbias_next needs dx16" in lib.vitb200_last_error()
    rc = lib.vitb200_cast16_colsum(stream(), a.data_ptr(), a.data_ptr(), a.data_ptr(), 2, 12, _lib.DT_F16, 0.0, 0, 0)
    assert rc == -1 and b"multiple of 8" in lib.vitb200_last_error()
    rc = lib.vitb200_gelu_fwd(stream(), a.data_ptr(), a.data_ptr(), 8, _lib.DT_F16, 1.0, 0, 0)
    assert rc == -1 and b"[0, 1)" in lib.vitb200_last_error()
    rc = lib.vitb200_pool_layernorm_bwd(stream(), a.data_ptr(), a.data_ptr(), a.data_ptr(), a.data_ptr(), a.data_ptr(),
                                        a.data_ptr(), a.data_ptr(), 1, 1, 64, 2, 1e-6)
    assert rc == -1 and b"pool" in lib.vitb200_last_error()
    rc = lib.vitb200_token_grads(stream(), a.data_ptr(), a.data_ptr(), None, a.data_ptr(), 1, 1, 64, 1)
    assert rc == -1 and b"null" in lib.vitb200_last_error()


# ================================================================ C. every leaf at the size that is trained
@pytest.mark.parametrize("precision,tol", [("fp16", 3e-2), ("bf16", 8e-2)])
def test_every_leaf_vit_b16_batch_256(precision, tol):
    """Full ViT-B/16 at batch 256 with wrt='both': every parameter leaf and the image gradient against float64 autograd
    on the device (_bwd_ref.vjp_on_device, 16 images per chunk), as max|g - g_ref| / max|g_ref| at the bounds the
    end-to-end tests use (fp16: that of the full-depth ViT-B/16 check, bf16: that of every bf16 check)."""
    cfg = dict(C2)
    variables = perturb_params(init_params(seed=71, **cfg), seed=72)
    img = images_for(cfg, 256, seed=73)
    dl = (np.random.default_rng(74).standard_normal((256, 1000)) / 16).astype(np.float32)
    eng = Engine(precision=precision, max_batch=256, **cfg)
    eng.load_params(variables)
    logits = eng.train_forward(torch.as_tensor(img, device="cuda")).cpu().numpy()
    dimg = eng.backward(torch.as_tensor(dl, device="cuda"), wrt="both").cpu().numpy()
    got = eng.grads()
    eng.close()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    want_logits, want, want_dimg = R.vjp_on_device(variables, img, dl, chunk=16, **cfg)
    torch.cuda.synchronize()
    print(f"\nfloat64 reference, ViT-B/16 batch 256: {time.perf_counter() - t0:.1f} s, "
          f"peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
    rel = lambda a, b: float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-30))
    assert rel(logits, want_logits) < (2e-2 if precision == "fp16" else 5e-2)
    ref = flatten_params({"params": want})
    assert set(got) == set(ref)
    errs = {k: rel(got[k], ref[k]) for k in ref}
    errs["images"] = rel(dimg, want_dimg)
    worst = max(errs, key=errs.get)
    print("worst leaves:", sorted(errs.items(), key=lambda kv: -kv[1])[:4])
    assert errs[worst] < tol, (worst, errs[worst])
