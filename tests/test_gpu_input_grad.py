"""Gradients with respect to the input images on a real B200: the patchify adjoint kernel, the image gradient of the
whole backward pass against float64 autograd (``tests/_input_grad_oracle.py``) or central differences (SimpleViT),
the exact properties of the image-only backward at ViT-B/16, and the errors of the new entry points."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import simple_vit_numpy
from vit_flax_b200 import SimpleViT, ViT, _lib, init_params, perturb_params
from vit_flax_b200._lib import VitB200Error
from vit_flax_b200.engine import Engine
from vit_flax_b200.params import flatten_params
from vit_flax_b200.runtime import clear_cache
from vit_flax_b200.simple_vit import clear_cache as clear_simple_cache
from _input_grad_oracle import vit_vjp_images
from _util import C2, TINY, images_for

pytestmark = pytest.mark.gpu

# a tiny mean-pool config the backward pass is built for (TINY_MEAN has heads 1 / dim 64: identity to_out)
TINY_MEAN2 = dict(image_size=(16, 32), patch_size=(8, 16), num_classes=16, dim=128, depth=1, heads=2, mlp_dim=64)
H14 = dict(image_size=224, patch_size=14, num_classes=1000, dim=1280, depth=1, heads=16, mlp_dim=5120)   # T = 257, K0 = 588
TOL = {"fp16": 2e-2, "bf16": 8e-2}


@pytest.fixture(scope="module")
def lib(lib_built):
    assert lib_built.vitb200_device_count() >= 1, "no sm_100 device"
    return lib_built


@pytest.fixture(autouse=True)
def _fresh_cache():
    yield
    clear_cache()
    clear_simple_cache()
    torch.cuda.empty_cache()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def rel_err(got, want):
    want = np.asarray(want, dtype=np.float64)
    return float(np.abs(np.asarray(got, dtype=np.float64) - want).max() / max(np.abs(want).max(), 1e-30))


# ---------------------------------------------------------------- unpatchify
def _patches_np(img, ph, pw, nchw):
    """'b h w (p1 p2 c)' feature order of vit.py:146 / simple_vit.py:125 -> [b, Np, K0]."""
    if nchw:
        b, c, H, W = img.shape
        x = img.reshape(b, c, H // ph, ph, W // pw, pw).transpose(0, 2, 4, 3, 5, 1)
    else:
        b, H, W, c = img.shape
        x = img.reshape(b, H // ph, ph, W // pw, pw, c).transpose(0, 1, 3, 2, 4, 5)
    return x.reshape(b, (H // ph) * (W // pw), ph * pw * c)


@pytest.mark.parametrize("cls_slot", [0, 1])
@pytest.mark.parametrize("nchw", [0, 1])
@pytest.mark.parametrize("H,W,C,ph,pw", [(224, 224, 3, 16, 16), (224, 224, 3, 14, 14), (224, 224, 3, 7, 7),
                                         (64, 64, 1, 16, 16), (64, 32, 4, 16, 16), (48, 80, 3, 16, 8), (32, 64, 3, 8, 16)])
def test_unpatchify_inverts_patchify(lib, H, W, C, ph, pw, nchw, cls_slot):
    """patchify_tokens (fp32) then unpatchify gives the images back bit for bit; the patch matrix equals the numpy
    reshape, and the rows / columns unpatchify must not read (class-token slots, K padding) hold NaN."""
    b = 3
    K0 = ph * pw * C
    Kpad = -(-K0 // 64) * 64
    Np = (H // ph) * (W // pw)
    shape = (b, C, H, W) if nchw else (b, H, W, C)
    img = torch.randn(shape, generator=torch.Generator().manual_seed(H + W + C + ph)).cuda()
    patches = torch.full((b * (Np + cls_slot), Kpad), float("nan"), device="cuda")
    _lib.check(lib.vitb200_patchify_tokens(stream(), img.data_ptr(), patches.data_ptr(), b, H, W, C, ph, pw, Kpad,
                                           _lib.DT_F32, nchw, cls_slot))
    p = patches.view(b, Np + cls_slot, Kpad)[:, cls_slot:, :K0].cpu().numpy()
    np.testing.assert_array_equal(p, _patches_np(img.cpu().numpy(), ph, pw, nchw))
    patches.view(b, Np + cls_slot, Kpad)[:, cls_slot:, K0:] = float("nan")      # pad columns: never read
    back = torch.full(shape, 7.0, device="cuda")
    _lib.check(lib.vitb200_unpatchify(stream(), patches.data_ptr(), back.data_ptr(), b, H, W, C, ph, pw, Kpad, nchw, cls_slot))
    torch.cuda.synchronize()
    assert torch.equal(back, img)


def test_unpatchify_of_an_arbitrary_matrix_is_the_numpy_inverse(lib):
    b, H, W, C, ph, pw = 2, 42, 28, 3, 7, 7
    K0, Kpad = ph * pw * C, 192
    Np = (H // ph) * (W // pw)
    g = torch.Generator().manual_seed(3)
    for nchw in (0, 1):
        patches = torch.randn((b * (Np + 1), Kpad), generator=g).cuda()
        out = torch.empty((b, C, H, W) if nchw else (b, H, W, C), device="cuda")
        _lib.check(lib.vitb200_unpatchify(stream(), patches.data_ptr(), out.data_ptr(), b, H, W, C, ph, pw, Kpad, nchw, 1))
        torch.cuda.synchronize()
        feats = patches.view(b, Np + 1, Kpad)[:, 1:, :K0].cpu().numpy()
        np.testing.assert_array_equal(_patches_np(out.cpu().numpy(), ph, pw, nchw), feats)


# ---------------------------------------------------------------- end to end
def _check_dx(cfg, precision, batch, seed, pool="cls", drop=0.0, max_batch=None):
    variables = perturb_params(init_params(seed=seed, **cfg), seed=seed + 1)
    img = images_for(cfg, batch, seed=seed + 2)
    dl = np.random.default_rng(seed + 3).standard_normal((batch, cfg["num_classes"])).astype(np.float32)
    kw = dict(pool=pool)
    if drop:
        kw.update(dropout=drop, emb_dropout=drop)
    eng = Engine(precision=precision, max_batch=max_batch or batch, **kw, **cfg)
    eng.load_params(variables)
    key = 0x5EED
    if drop:
        eng.set_dropout_key(key)
    x = torch.as_tensor(img, device="cuda")
    eng.train_forward(x)
    dx = eng.backward(torch.as_tensor(dl, device="cuda"), wrt="input").cpu().numpy()
    okw = dict(kw, dropout_key=key) if drop else kw
    _, _, want = vit_vjp_images(variables, img, dl, **okw, **cfg)
    assert dx.shape == img.shape and np.isfinite(dx).all()
    err = rel_err(dx, want)
    assert err <= TOL[precision], err
    eng.close()
    return err


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("cfg,pool", [(TINY, "cls"), (TINY_MEAN2, "mean")])
def test_image_gradient_tiny(cfg, pool, precision):
    _check_dx(cfg, precision, 5, 100, pool=pool, max_batch=7)


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_image_gradient_with_dropout_replays_the_masks(precision):
    cfg = dict(image_size=32, patch_size=8, num_classes=16, dim=128, depth=2, heads=2, mlp_dim=256)
    _check_dx(cfg, precision, 4, 200, drop=0.1)


def test_image_gradient_vit_b16_geometry():
    _check_dx(dict(C2, depth=2), "fp16", 2, 300)


def test_image_gradient_vit_h14_geometry():
    """T = 257 (the streamed attention adjoint) and K0 = 588 (padded to 640 for the patch-feature GEMM)."""
    _check_dx(H14, "fp16", 2, 400)


def test_vjp_surface_both_and_cuda_tensors():
    """ViT.vjp(wrt=...): 'params' unchanged, 'input' -> dx, 'both' -> (tree, dx); numpy in -> numpy out, CUDA in ->
    CUDA out; the loss scaling of tiny cotangents is undone on dx too."""
    cfg = dict(TINY)
    v = ViT(**cfg)
    variables = perturb_params(init_params(seed=41, **cfg), seed=42)
    img = images_for(cfg, 3, seed=43)
    dl = (np.random.default_rng(44).standard_normal((3, cfg["num_classes"])) * 1e-7).astype(np.float32)
    _, want_g, want_dx = vit_vjp_images(variables, img, dl, **cfg)
    _, f = v.vjp(variables, img, wrt="input")
    dx = f(dl)
    assert isinstance(dx, np.ndarray) and dx.shape == img.shape and dx.dtype == np.float32
    assert rel_err(dx, want_dx) < 2e-2
    _, f = v.vjp(variables, img, wrt="both")
    g, dx2 = f(dl)
    np.testing.assert_array_equal(dx2, dx)
    got, ref = flatten_params(g), flatten_params({"params": want_g})
    assert set(got) == set(ref) and all(rel_err(got[k], ref[k]) < 2e-2 for k in ref)
    _, f = v.vjp(variables, img)
    assert set(flatten_params(f(dl))) == set(ref)
    xc = torch.as_tensor(img, device="cuda")
    _, f = v.vjp(variables, xc, wrt="input")
    dxc = f(torch.as_tensor(dl, device="cuda"))
    assert dxc.is_cuda and dxc.dtype == torch.float32 and tuple(dxc.shape) == img.shape
    np.testing.assert_array_equal(dxc.cpu().numpy(), dx)


def test_simple_vit_image_gradient_matches_finite_differences_of_the_oracle():
    """SimpleViT (NCHW, no class token): dimg at its largest entries and at random pixels against central
    differences of the float64 numpy oracle."""
    cfg = dict(image_size=(32, 64), patch_size=(8, 16), num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128)
    v = SimpleViT(**cfg)
    img = np.random.default_rng(5).standard_normal((3, 3, 32, 64)).astype(np.float32)
    params = v.init({"params": 6}, img)
    dl = np.random.default_rng(7).standard_normal((3, cfg["num_classes"]))
    _, f = v.vjp(params, img, wrt="input")
    dx = f(dl.astype(np.float32))
    assert dx.shape == img.shape and dx.dtype == np.float32
    scale = np.abs(dx).max()
    rng = np.random.default_rng(8)
    picks = [np.unravel_index(i, dx.shape) for i in np.argsort(np.abs(dx).ravel())[-6:]]
    picks += [tuple(int(rng.integers(0, s)) for s in dx.shape) for _ in range(10)]
    loss = lambda x: float((simple_vit_numpy.simple_vit_forward(params, x, **cfg) * dl).sum())
    for idx in picks:
        vals = []
        for sgn in (1, -1):
            x = img.astype(np.float64).copy()
            x[idx] += sgn * 1e-4
            vals.append(loss(x))
        fd = (vals[0] - vals[1]) / 2e-4
        assert abs(dx[idx] - fd) < 3e-2 * scale, (idx, dx[idx], fd)
    _, f = v.vjp(params, img, wrt="both")
    g, dx2 = f(dl.astype(np.float32))
    np.testing.assert_array_equal(dx2, dx)
    assert set(g["params"]) == set(params["params"])


# ---------------------------------------------------------------- exact properties at ViT-B/16
def test_image_gradient_properties_vit_b16_full_batch():
    """ViT-B/16, 12 layers, batch 256.  (1) dx of wrt='input' == dx of wrt='both' bit for bit (the dx chain is the
    same launches either way); (2) parameter gradients of 'both' == those of 'params' up to the order in which
    split-K partial sums and column-sum atomics land (two 'params' runs differ by as much); (3) an image whose
    cotangent row is zero gets dx == 0 exactly; (4) dx is linear in the cotangent (to the fp16 floor, below)."""
    cfg = dict(C2)
    eng = Engine(precision="fp16", max_batch=256, **cfg)
    eng.load_params(perturb_params(init_params(seed=61, **cfg), seed=62))
    x = torch.as_tensor(images_for(cfg, 256, seed=63), device="cuda")
    dl = torch.as_tensor((np.random.default_rng(64).standard_normal((256, 1000)) / 16).astype(np.float32), device="cuda")
    zero_rows = [0, 17, 255]
    dl[zero_rows] = 0.0
    eng.train_forward(x)
    dx_in = eng.backward(dl, wrt="input").clone()
    with pytest.raises(VitB200Error, match="did not compute parameter gradients"):
        eng.grads_flat()
    dx_both = eng.backward(dl, wrt="both").clone()
    g_both = eng.grads_flat().clone()
    eng.backward(dl, wrt="params")
    g_p1 = eng.grads_flat().clone()
    eng.backward(dl, wrt="params")
    g_p2 = eng.grads_flat().clone()
    dx_twice = eng.backward((2 * dl).contiguous(), wrt="input").clone()
    assert torch.isfinite(dx_in).all() and dx_in.abs().max() > 0
    assert torch.equal(dx_in, dx_both)
    spread = float((g_p1 - g_p2).abs().max())
    ref = float(g_p1.abs().max())
    assert float((g_both - g_p1).abs().max()) <= max(2 * spread, 1e-5 * ref), (float((g_both - g_p1).abs().max()), spread, ref)
    for r in zero_rows:
        assert torch.count_nonzero(dx_in[r]) == 0, r
    # doubling is exact in fp32 and for normal fp16 values, not for the fp16-subnormal entries of the 16-bit cotangents
    # (|x| < 6.1e-5), so the map is linear to the 16-bit format's floor here, the bound the parameter gradients'
    # linearity test uses; ViT.vjp's power-of-two cotangent scaling makes it exact at that surface
    assert float((dx_twice - 2 * dx_in).abs().max()) <= 5e-3 * float((2 * dx_in).abs().max())
    eng.close()


# ---------------------------------------------------------------- errors
def test_image_gradient_errors(lib):
    cfg = dict(TINY)
    v = ViT(**cfg)
    variables = perturb_params(init_params(seed=1, **cfg), seed=2)
    img = images_for(cfg, 2, seed=3)
    dl = np.ones((2, cfg["num_classes"]), np.float32)
    with pytest.raises(VitB200Error, match="bf16/fp16"):
        v.vjp(variables, img, wrt="input", precision="fp32")
    # grads() after an image-only backward
    eng = Engine(precision="fp16", max_batch=2, **cfg)
    eng.load_params(variables)
    x = torch.as_tensor(img, device="cuda")
    d = torch.as_tensor(dl, device="cuda")
    eng.train_forward(x)
    eng.backward(d, wrt="input")
    for call in (eng.grads, lambda: eng.grad_tensor("cls"), eng.grads_flat):
        with pytest.raises(VitB200Error, match="did not compute parameter gradients"):
            call()
    eng.backward(d)
    assert np.isfinite(eng.grads()["cls"]).all()
    # the C entry point's own argument checks
    dimg = torch.empty_like(x)
    h = eng.handle
    for wrt, ptr in ((0, dimg.data_ptr()), (4, dimg.data_ptr()), (_lib.GRAD_IMAGES, None), (_lib.GRAD_PARAMS | _lib.GRAD_IMAGES, None)):
        assert lib.vitb200_backward_ex(h, stream(), d.data_ptr(), 2, wrt, ptr) == -1, wrt    # VITB200_ERR_INVALID
    assert lib.vitb200_backward_ex(h, stream(), d.data_ptr(), 2, _lib.GRAD_IMAGES, dimg.data_ptr()) == 0
    with pytest.raises(ValueError, match="wrt"):
        eng.backward(d, wrt="everything")
    eng.close()
    # a vjp_fn whose forward went stale is refused for wrt='input' too
    _, f = v.vjp(variables, img, wrt="input")
    v.apply(variables, images_for(cfg, 2, seed=4))
    with pytest.raises(RuntimeError, match="another forward"):
        f(dl)
