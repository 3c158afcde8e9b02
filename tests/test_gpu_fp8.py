"""precision='fp8' on a real B200: the E4M3 GEMM, LayerNorm and weight-quantisation kernels through the C ABI, and the
forward through the public API against the emulation in tests/_fp8_oracle.py and the fp32 oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import vit_torch
from vit_flax_b200 import SimpleViT, ViT, _lib
from vit_flax_b200.engine import Engine
from vit_flax_b200.params import init_params, perturb_params
from vit_flax_b200.runtime import clear_cache
from _fp8_oracle import decode_e4m3, e4m3_codes, quantize_weight, vit_forward_fp8
from _util import C2, TINY, TINY_MEAN, images_for

pytestmark = pytest.mark.gpu

# every finite E4M3 value in increasing order: two codes are one step apart when their values are neighbours here
_VALUES = np.unique(decode_e4m3(np.array([c for c in range(256) if (c & 0x7F) != 0x7F], np.uint8)))


@pytest.fixture(scope="module")
def lib(lib_built):
    assert lib_built.vitb200_device_count() >= 1, "no sm_100 device"
    return lib_built


@pytest.fixture(autouse=True)
def _fresh():
    yield
    clear_cache()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.asarray(a)).to("cuda", dtype).contiguous()


def random_codes(rng, shape):
    """Random finite E4M3 codes (no NaN), both signs, spread over the whole exponent range."""
    c = rng.integers(0, 256, shape, dtype=np.uint8)
    return np.where((c & 0x7F) == 0x7F, c & 0xF0, c).astype(np.uint8)


def check_codes(got, ref, bound, what):
    """E4M3 codes ``got`` against the float64 reference values ``ref``: equal to their rounding, except one step where
    ``ref`` lies within ``bound`` (the device's fp32 error) of the midpoint between the two neighbouring values."""
    want = e4m3_codes(ref.astype(np.float32))
    g, w = decode_e4m3(got), decode_e4m3(want)
    bad = g != w
    if bad.any():
        ig, iw = np.searchsorted(_VALUES, g[bad]), np.searchsorted(_VALUES, w[bad])
        mid = (g[bad] + w[bad]) / 2
        ok = (np.abs(ig - iw) == 1) & (np.abs(ref[bad] - mid) <= np.broadcast_to(bound, ref.shape)[bad])
        assert ok.all(), f"{what}: {int((~ok).sum())} codes off by more than a midpoint rounding " \
                         f"(first: got {g[bad][~ok][:4]}, want {w[bad][~ok][:4]}, ref {ref[bad][~ok][:4]})"
    print(f"[fp8 codes] {what}: {int(bad.sum())} of {bad.size} one step off at a midpoint")


# N a multiple of 16 (E4M3 output rows of a 16-byte pitch), ragged against the 64- and 256-column tiles
GEMM_CASES = [(128, 256, 64), (300, 272, 208), (1576, 2304, 768), (600, 784, 3072), (40, 3072, 768)]


@pytest.mark.parametrize("M,N,K", GEMM_CASES)
@pytest.mark.parametrize("epi", [_lib.EPI_STORE_16, _lib.EPI_BIAS_GELU_E4M3, _lib.EPI_BIAS_RESID_F32, _lib.EPI_BIAS_F32])
@pytest.mark.parametrize("cta_group", ["1", "2", "64"])
def test_gemm_e4m3_epilogues(lib, M, N, K, epi, cta_group, monkeypatch):
    """K 64 is shorter than one 128-element k-block, 208 ragged; M and N ragged.  Operands are exact E4M3 codes, so the
    float64 product of the decoded values is the reference and the only error is fp32 accumulation (1e-5 of the row's
    sum of |a||w|) plus the output rounding."""
    monkeypatch.setenv("VITB200_GEMM_CTA_GROUP", cta_group)
    rng = np.random.default_rng(M + N + K + epi)
    a8, w8 = random_codes(rng, (M, K)), random_codes(rng, (N, K))
    a, w = decode_e4m3(a8), decode_e4m3(w8)
    ws = rng.uniform(0.5, 2.0, N).astype(np.float32) / np.float32(np.sqrt(K) * 64.0)
    bias = (rng.standard_normal(N) * 0.5).astype(np.float32)
    acc = (a @ w.T) * ws.astype(np.float64)
    mag = (np.abs(a) @ np.abs(w).T) * ws.astype(np.float64)
    A, Wt, WS, B = dev(a8, torch.uint8), dev(w8, torch.uint8), dev(ws), dev(bias)
    if epi == _lib.EPI_STORE_16:
        out = torch.zeros((M, N), dtype=torch.float16, device="cuda")
    elif epi == _lib.EPI_BIAS_GELU_E4M3:
        out = torch.zeros((M, N), dtype=torch.uint8, device="cuda")
    else:
        resid = (rng.standard_normal((M, N))).astype(np.float32)
        out = dev(resid) if epi == _lib.EPI_BIAS_RESID_F32 else torch.zeros((M, N), device="cuda")
    _lib.check(lib.vitb200_gemm_tc_e4m3(stream(), A.data_ptr(), Wt.data_ptr(), WS.data_ptr(), B.data_ptr(),
                                        out.data_ptr(), M, N, K, epi))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    tol = 1e-5 * mag + 1e-30
    if epi == _lib.EPI_STORE_16:
        assert np.all(np.abs(got.astype(np.float64) - acc) <= tol + 2.0 ** -11 * np.abs(acc) + 2.0 ** -24)
    elif epi == _lib.EPI_BIAS_GELU_E4M3:
        y = acc + bias
        gelu = 0.5 * y * (1.0 + np.tanh(0.7978845608028654 * (y + 0.044715 * y ** 3)))
        # tanh.approx.f32: relative error below 2^-10.9; the GELU's slope is below 1.13
        check_codes(got, gelu, 1.2 * tol + 0.5 * np.abs(y) * 2.0 ** -10 + 1e-7, f"gelu M={M} N={N} K={K} mode {cta_group}")
    elif epi == _lib.EPI_BIAS_RESID_F32:
        assert np.all(np.abs(got - (resid + acc + bias)) <= tol + 1e-6 * (np.abs(resid) + np.abs(bias) + 1))
    else:
        assert np.all(np.abs(got - (acc + bias)) <= tol + 1e-6 * (np.abs(bias) + 1))


def test_gemm_e4m3_rejections(lib):
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    assert lib.vitb200_gemm_tc_e4m3(stream(), p, p, p, p, p, 128, 256, 200, _lib.EPI_STORE_16) == -1   # K % 16
    assert lib.vitb200_gemm_tc_e4m3(stream(), p, p, p, p, p, 128, 264, 256, _lib.EPI_BIAS_GELU_E4M3) == -1  # N % 16
    assert lib.vitb200_gemm_tc_e4m3(stream(), p, p, p, p, p, 128, 256, 256, _lib.EPI_BIAS_GELU_16) == -4
    assert lib.vitb200_gemm_tc_e4m3(stream(), p, p, None, p, p, 128, 256, 256, _lib.EPI_STORE_16) == -1
    # the other launchers that share the dtype switch keep rejecting E4M3
    assert lib.vitb200_patchify(stream(), p, p, 1, 32, 32, 3, 8, 8, 192, _lib.DT_E4M3) == -1
    assert lib.vitb200_pool_layernorm(stream(), p, p, p, p, 1, 4, 64, 0, _lib.DT_E4M3) == -1


@pytest.mark.parametrize("rows,dim", [(1000, 768), (37, 1024), (5, 200)])
def test_layernorm_e4m3_output(lib, rows, dim):
    rng = np.random.default_rng(rows + dim)
    x = (rng.standard_normal((rows, dim)) * 3 + rng.standard_normal((rows, 1))).astype(np.float32)
    g = rng.uniform(0.2, 3.0, dim).astype(np.float32)
    b = (rng.standard_normal(dim) * 0.5).astype(np.float32)
    y = torch.zeros((rows, dim), dtype=torch.uint8, device="cuda")
    X, G, Bv = dev(x), dev(g), dev(b)
    _lib.check(lib.vitb200_layernorm(stream(), X.data_ptr(), G.data_ptr(), Bv.data_ptr(), y.data_ptr(), rows, dim, _lib.DT_E4M3))
    torch.cuda.synchronize()
    xd = x.astype(np.float64)
    ref = (xd - xd.mean(1, keepdims=True)) / np.sqrt(xd.var(1, keepdims=True) + 1e-6) * g + b
    check_codes(y.cpu().numpy(), ref, 1e-5 * (np.abs(ref) + 1.0), f"layernorm {rows}x{dim}")


@pytest.mark.parametrize("K,N,Kpad", [(768, 2304, 768), (200, 40, 256), (3072, 768, 3072), (64, 1000, 64)])
def test_quantize_weight_bit_exact(lib, K, N, Kpad):
    rng = np.random.default_rng(K + N)
    W = (rng.standard_normal((K, N)) * rng.uniform(0.001, 2.0, N)).astype(np.float32)
    W[:, 3] = 0.0
    Wt = torch.full((N, Kpad), 0xAB, dtype=torch.uint8, device="cuda")
    scale = torch.zeros(N, device="cuda")
    Wd = dev(W)
    _lib.check(lib.vitb200_quantize_weight_e4m3(stream(), Wd.data_ptr(), Wt.data_ptr(), scale.data_ptr(), K, N, Kpad))
    torch.cuda.synchronize()
    w8, s = quantize_weight(W)
    np.testing.assert_array_equal(scale.cpu().numpy(), s.numpy())
    got = Wt.cpu().numpy()
    np.testing.assert_array_equal(got[:, :K], e4m3_codes(w8.numpy().T))
    assert np.all(got[:, K:] == 0)


# ---- end to end -------------------------------------------------------------------------------------------------------
def _bounds(got, emu, want):
    """The bf16 criterion of DESIGN.md section 5 with F = |emulation - fp32 oracle| on the same inputs."""
    F = float(np.abs(emu - want).max())
    e_or, e_emu = float(np.abs(got - want).max()), float(np.abs(got - emu).max())
    return F, e_or, e_emu


def _check_vit(cfg, batch, pool="cls", depth=None, perturb=True):
    cfg = dict(cfg, depth=depth) if depth is not None else cfg
    variables = init_params(seed=1, **cfg)
    if perturb:
        variables = perturb_params(variables, seed=2)
    img = images_for(cfg, batch, seed=0)
    got = ViT(pool=pool, **cfg).apply(variables, img, precision="fp8")
    want = vit_torch.vit_forward(vit_torch.tree_to_torch(variables), img, pool=pool, **cfg).numpy()
    emu = vit_forward_fp8(variables, img, pool=pool, **cfg)
    F, e_or, e_emu = _bounds(got, emu, want)
    print(f"[fp8 parity] depth={cfg['depth']} dim={cfg['dim']} pool={pool} batch={batch}: |gpu-oracle| {e_or:.4f} "
          f"(bound {max(2e-2, 1.25 * F):.4f}), |gpu-emulation| {e_emu:.4f} (bound {max(2e-2, F):.4f}), F {F:.4f}")
    assert e_or <= max(2e-2, 1.25 * F)
    assert e_emu <= max(2e-2, F)


@pytest.mark.parametrize("cfg,pool", [(TINY, "cls"), (TINY_MEAN, "mean")])
def test_fp8_tiny(cfg, pool):
    _check_vit(cfg, 5, pool)


def test_fp8_vit_b16_reduced_depth():
    _check_vit(C2, 4, depth=2)


def test_fp8_vit_b16_full_depth():
    _check_vit(C2, 8)


def test_fp8_simple_vit_demo():
    cfg = dict(image_size=256, patch_size=32, num_classes=1000, dim=1024, depth=6, heads=16, mlp_dim=2048)
    v = SimpleViT(**cfg)
    img = np.random.default_rng(3).standard_normal((2, 3, 256, 256)).astype(np.float32)   # NCHW
    params = v.init({"params": 4}, img)
    got = v.apply(params, img, precision="fp8")
    tree = v._engine_tree(params)
    kw = dict(patch_size=32, dim=1024, depth=6, heads=16, pool="mean", cls_token=False, ln_eps=1e-5)
    nhwc = img.transpose(0, 2, 3, 1)
    want = vit_forward_fp8(tree, nhwc, rounding="none", **kw)
    emu = vit_forward_fp8(tree, nhwc, **kw)
    F, e_or, e_emu = _bounds(got, emu, want)
    print(f"[fp8 parity] SimpleViT demo: |gpu-oracle| {e_or:.4f}, |gpu-emulation| {e_emu:.4f}, F {F:.4f}")
    assert e_or <= max(2e-2, 1.25 * F)
    assert e_emu <= max(2e-2, F)


def test_fp8_vit_b16_batch_256_properties():
    """Top-1 agreement where the oracle's margin exceeds 2F, device == host path, run-to-run bits, independence of
    batch neighbours, apply_stream, and batch 1 through the captured graph."""
    cfg = C2
    variables = perturb_params(init_params(seed=1, **cfg), seed=2)
    img = images_for(cfg, 256, seed=0)
    v = ViT(**cfg)
    y_host = v.apply(variables, img, precision="fp8")
    x_dev = torch.as_tensor(img, device="cuda")
    y_dev = v.apply(variables, x_dev, precision="fp8")
    y_dev2 = v.apply(variables, x_dev, precision="fp8")
    np.testing.assert_array_equal(y_host, y_dev.cpu().numpy())
    assert torch.equal(y_dev, y_dev2)
    perm = np.random.default_rng(0).permutation(256)
    assert np.abs(v.apply(variables, img[perm], precision="fp8") - y_host[perm]).max() < 1e-4
    streamed = np.concatenate([o.copy() for o in v.apply_stream(variables, (img[i:i + 64] for i in range(0, 256, 64)),
                                                                precision="fp8")])
    np.testing.assert_array_equal(streamed, y_host)
    pt = vit_torch.tree_to_torch(variables)
    want = np.concatenate([vit_torch.vit_forward(pt, img[i:i + 32], **cfg).numpy() for i in range(0, 256, 32)])
    F = float(np.abs(vit_forward_fp8(variables, img[:16], **cfg) - want[:16]).max())
    top2 = np.sort(want, axis=1)[:, -2:]
    sure = (top2[:, 1] - top2[:, 0]) > 2 * F
    agree = (y_host.argmax(1) == want.argmax(1))[sure]
    print(f"[fp8 top-1] {int(sure.sum())} of 256 images with an oracle margin > 2F = {2 * F:.3f}: {int(agree.sum())} agree")
    assert agree.all()
    # batch 1: a captured graph (small batch); its bits equal the directly launched forward's
    eng = Engine(precision="fp8", max_batch=1, **cfg)
    eng.load_params(variables)
    x1 = x_dev[:1].contiguous()
    a = eng.forward(x1).clone()
    b = eng.forward(x1).clone()
    direct = torch.empty_like(a)
    eng.profile_forward(x1, out=direct)
    torch.cuda.synchronize()
    assert torch.equal(a, b) and torch.equal(a, direct)
    assert np.abs(a.cpu().numpy() - y_host[:1]).max() < 1e-4
    eng.close()


def test_fp8_error_paths():
    cfg = TINY
    variables = init_params(seed=1, **cfg)
    img = images_for(cfg, 2, seed=0)
    with pytest.raises(ValueError, match="dropout"):
        ViT(dropout=0.1, **cfg).apply(variables, img, rngs={"dropout": 0}, precision="fp8")
    with pytest.raises(ValueError, match="fp8"):
        ViT(**cfg).vjp(variables, img, precision="fp8")
    with pytest.raises(ValueError, match="fp8"):
        SimpleViT(image_size=32, patch_size=8, num_classes=8, dim=64, depth=1, heads=2, mlp_dim=128).vjp(
            {"params": {}}, np.zeros((1, 3, 32, 32), np.float32), precision="fp8")
    from vit_flax_b200 import adamw
    with pytest.raises(ValueError, match="fp16 or bf16"):
        ViT(**cfg).trainer(variables, adamw(1e-3), precision="fp8")
    with pytest.raises(ValueError, match="precision"):
        ViT(**cfg).apply(variables, img, precision="fp4")
    eng = Engine(precision="fp8", max_batch=2, **cfg)
    eng.load_params(variables)
    x = torch.as_tensor(img, device="cuda")
    for call in (lambda: eng.train_forward(x), lambda: eng.backward(torch.zeros((2, 8), device="cuda")),
                 lambda: eng.adamw_step(lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, weight_decay=0.0)):
        with pytest.raises(ValueError, match="fp8"):
            call()
    # the C ABI refuses the same on an fp8 handle
    lib, h = eng.lib, eng.handle
    out = torch.empty((2, 8), device="cuda")
    assert lib.vitb200_train_forward(h, stream(), x.data_ptr(), 2, out.data_ptr()) == -4
    assert lib.vitb200_backward(h, stream(), out.data_ptr(), 2) == -4
    assert lib.vitb200_adamw_step(h, stream(), C.byref(_lib.AdamW(lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, grad_scale=1.0))) == -4
    eng.close()
    cfg_c = _lib.Config(image_h=32, image_w=32, patch_h=8, patch_w=8, channels=3, num_classes=8, dim=64, depth=1, heads=2,
                        mlp_dim=128, pool=0, precision=_lib.PREC_FP8, max_batch=1, dropout=0.1)
    handle = C.c_void_p()
    assert lib.vitb200_create(C.byref(cfg_c), 0, C.byref(handle)) == -4
    cfg_c.dropout, cfg_c.precision = 0.0, 7
    assert lib.vitb200_create(C.byref(cfg_c), 0, C.byref(handle)) == -1
