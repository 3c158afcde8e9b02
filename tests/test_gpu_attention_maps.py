"""Attention maps on a real B200: ``attention_maps`` / ``vitb200_forward_attn`` leave the forward's logits and launches
alone, match the float64 oracle within the error floor of the operand format (tests/_attn_oracle.py), and hold the
exact properties of a softmax; the recompute kernel is also checked alone through the C ABI."""
import ctypes as C

import numpy as np
import pytest
import torch

from vit_flax_b200 import SimpleViT, ViT, _lib
from vit_flax_b200.engine import Engine, launch_count
from vit_flax_b200.params import init_params, perturb_params
from vit_flax_b200.runtime import clear_cache
from vit_flax_b200 import simple_vit as _simple_vit
from _attn_oracle import error_floor, simple_vit_attention_maps, tolerance, vit_attention_maps
from _util import C2, C4, C5, TINY, TINY_MEAN, images_for, load_golden

pytestmark = pytest.mark.gpu

T65 = dict(image_size=128, patch_size=16, num_classes=10, dim=256, depth=2, heads=4, mlp_dim=512)   # 64 patches + cls


@pytest.fixture(scope="module")
def lib(lib_built):
    assert lib_built.vitb200_device_count() >= 1, "no sm_100 device"
    return lib_built


@pytest.fixture(autouse=True)
def _fresh():
    yield
    clear_cache()
    _simple_vit.clear_cache()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def check_against_oracle(got, variables, images, cfg, precision, what, **kw):
    """GPU maps against the float64 oracle, within FLOOR_MULT x the emulated error floor of the format."""
    fmt = {"fp16": "fp16", "bf16": "bf16", "fp8": "e4m3"}[precision]
    _, exact = vit_attention_maps(variables, images, **cfg, **kw)
    _, emu = vit_attention_maps(variables, images, rounding=fmt, **cfg, **kw)
    floor = error_floor(emu, exact)
    err = float(np.abs(got.astype(np.float64) - exact).max())
    print(f"[attention maps] {what} {precision}: max |P - P_ref| {err:.2e}, floor {floor:.2e}, tol {tolerance(floor):.2e}")
    assert got.shape == exact.shape
    assert err <= tolerance(floor), f"{what} {precision}: {err:.3e} > {tolerance(floor):.3e}"
    return exact


# ---------------------------------------------------------------- the forward is untouched
@pytest.mark.parametrize("precision,dropout", [("fp16", 0.0), ("bf16", 0.0), ("fp8", 0.0), ("fp16", 0.1), ("bf16", 0.1)])
def test_logits_and_launches_of_the_forward_are_untouched(lib, precision, dropout):
    """ViT-B/16 at batch 256: the fold schedule (dropout 0, fp16 / bf16) and the LayerNorm-kernel schedule (fp8, and
    dropout > 0).  The recording forward's logits are apply's bit for bit, it adds one launch per recorded layer, and a
    plain apply launches what it launched before."""
    v = ViT(dropout=dropout, **C2)
    variables = perturb_params(init_params(seed=1, **C2), seed=2)
    x = torch.as_tensor(images_for(C2, 256, seed=3), device="cuda")
    rngs = {"dropout": 1234} if dropout else None
    want = v.apply(variables, x, rngs, precision=precision)
    torch.cuda.synchronize()
    n0 = launch_count()
    v.apply(variables, x, rngs, precision=precision)
    plain = launch_count() - n0
    layers = [11, 0, 5]
    n0 = launch_count()
    logits, maps = v.attention_maps(variables, x, rngs, layers=layers, precision=precision)
    recording = launch_count() - n0
    torch.cuda.synchronize()
    assert torch.equal(logits, want)
    assert recording == plain + len(layers)
    n0 = launch_count()
    again = v.apply(variables, x, rngs, precision=precision)
    assert launch_count() - n0 == plain
    assert torch.equal(again, want)
    assert maps.shape == (256, 3, 12, 197, 197) and maps.is_cuda
    assert float((maps.sum(-1) - 1).abs().max()) < 1e-5


def test_full_size_vit_b16_all_layers(lib):
    """ViT-B/16, batch 256, all 12 layers: 5.7 GB of maps."""
    v = ViT(**C2)
    variables = perturb_params(init_params(seed=1, **C2), seed=2)
    x = torch.as_tensor(images_for(C2, 256, seed=4), device="cuda")
    want = v.apply(variables, x)
    logits, maps = v.attention_maps(variables, x)
    torch.cuda.synchronize()
    assert maps.shape == (256, 12, 12, 197, 197) and maps.dtype == torch.float32
    assert torch.equal(logits, want)
    assert float((maps.sum(-1) - 1).abs().max()) < 1e-5
    assert bool(torch.isfinite(maps).all()) and float(maps.min()) >= 0 and float(maps.max()) <= 1


# ---------------------------------------------------------------- against the oracle
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("name,cfg", [("tiny_cls.npz", TINY), ("tiny_mean.npz", dict(TINY_MEAN, pool="mean"))])
def test_golden_configs_against_the_oracle(lib, name, cfg, precision):
    variables, meta = load_golden(name)
    logits, maps = ViT(**cfg).attention_maps(variables, meta["images"], precision=precision)
    assert isinstance(maps, np.ndarray) and maps.dtype == np.float32
    check_against_oracle(maps, variables, meta["images"], cfg, precision, name)


GEOMETRIES = [("vit_b16_depth2", dict(C2, depth=2), 2),          # T = 197
              ("vit_h14_depth2", dict(C4, depth=2), 2),          # T = 257: streamed keys, three key blocks
              ("vit_512px_depth1", dict(C5, depth=1), 1),        # T = 1025: nine key blocks
              ("t65", T65, 3)]                                   # T = 65: one key block, a 65-row query tile


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("what,cfg,batch", GEOMETRIES)
def test_geometries_against_the_oracle(lib, what, cfg, batch, precision):
    variables = perturb_params(init_params(seed=5, **cfg), seed=6)
    img = images_for(cfg, batch, seed=7)
    logits, maps = ViT(**cfg).attention_maps(variables, img, precision=precision)
    exact = check_against_oracle(maps, variables, img, cfg, precision, what)
    # zeros only where the oracle underflows fp32
    zero = maps == 0
    assert not zero.any() or float(exact[zero].max()) < 2.0 ** -120


def test_fp8_against_the_oracle(lib):
    """fp8 runs the LayerNorm-kernel schedule with E4M3 to_qkv operands and fp16 q / k: the floor is the E4M3 one."""
    cfg = T65
    variables = perturb_params(init_params(seed=5, **cfg), seed=6)
    img = images_for(cfg, 3, seed=7)
    _, maps = ViT(**cfg).attention_maps(variables, img, precision="fp8")
    check_against_oracle(maps, variables, img, cfg, "fp8", "t65")
    assert np.abs(maps.sum(-1) - 1).max() < 1e-5


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_simple_vit_against_the_oracle(lib, precision):
    cfg = dict(image_size=224, patch_size=16, num_classes=10, dim=256, depth=2, heads=4, mlp_dim=512)
    v = SimpleViT(**cfg)
    img = np.random.default_rng(0).standard_normal((2, 3, 224, 224)).astype(np.float32)
    variables = v.init(1, img)
    logits, maps = v.attention_maps(variables, img, precision=precision)
    assert maps.shape == (2, 2, 4, 196, 196)
    np.testing.assert_array_equal(logits, v.apply(variables, img, precision=precision))
    fmt = "fp16" if precision == "fp16" else "bf16"
    _, exact = simple_vit_attention_maps(variables, img, **cfg)
    floor = error_floor(simple_vit_attention_maps(variables, img, rounding=fmt, **cfg)[1], exact)
    err = float(np.abs(maps - exact).max())
    print(f"[attention maps] simple_vit {precision}: {err:.2e}, floor {floor:.2e}")
    assert err <= tolerance(floor)


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_dropout_maps_are_those_of_the_dropped_forward(lib, precision):
    cfg = T65
    variables = perturb_params(init_params(seed=7, **cfg), seed=8)
    img = images_for(cfg, 3, seed=9)
    v = ViT(dropout=0.1, **cfg)
    key = 0xC0FFEE
    logits, maps = v.attention_maps(variables, img, {"dropout": key}, precision=precision)
    np.testing.assert_array_equal(logits, v.apply(variables, img, {"dropout": key}, precision=precision))
    check_against_oracle(maps, variables, img, cfg, precision, "dropout 0.1", dropout=0.1, dropout_key=key)
    _, other = v.attention_maps(variables, img, {"dropout": key + 1}, precision=precision)
    assert np.abs(other[:, 1] - maps[:, 1]).max() > 1e-3            # layer 1 sees another dropped stream


# ---------------------------------------------------------------- exact properties
def test_exact_properties(lib):
    cfg = dict(C2, depth=4)
    v = ViT(**cfg)
    variables = perturb_params(init_params(seed=11, **cfg), seed=12)
    x = torch.as_tensor(images_for(cfg, 4, seed=13), device="cuda")
    logits, maps = v.attention_maps(variables, x)
    assert logits.is_cuda and maps.is_cuda and maps.shape == (4, 4, 12, 197, 197)
    assert float((maps.sum(-1) - 1).abs().max()) < 1e-5
    assert bool(torch.isfinite(maps).all()) and float(maps.min()) >= 0 and float(maps.max()) <= 1
    # run to run
    _, again = v.attention_maps(variables, x)
    assert torch.equal(again, maps)
    # a subset, in the order asked for, is the same bits as those slices of all layers
    _, sub = v.attention_maps(variables, x, layers=[3, 0])
    assert torch.equal(sub, maps[:, [3, 0]])
    # an image's maps do not depend on its batch neighbours
    y = x.clone()
    y[1:] = torch.as_tensor(images_for(cfg, 3, seed=14), device="cuda")
    _, other = v.attention_maps(variables, y)
    assert torch.equal(other[0], maps[0]) and not torch.equal(other[1], maps[1])
    # host in, numpy out
    hl, hm = v.attention_maps(variables, x.cpu().numpy(), layers=[2])
    assert isinstance(hl, np.ndarray) and isinstance(hm, np.ndarray)
    np.testing.assert_array_equal(hm, maps[:, [2]].cpu().numpy())
    np.testing.assert_array_equal(hl, logits.cpu().numpy())
    # a caller's buffer
    eng = Engine(**cfg, precision="fp16", max_batch=4)
    eng.load_params(variables)
    buf = torch.full((4, 1, 12, 197, 197), -1.0, device="cuda")
    _, got = eng.forward_attn(x, [1], maps=buf)
    assert got is buf and torch.equal(buf, maps[:, [1]])
    eng.close()


@pytest.mark.parametrize("dtype", [_lib.DT_F16, _lib.DT_BF16])
@pytest.mark.parametrize("T", [65, 197, 257, 1025])
def test_kernels_alone_on_random_qkv(lib, T, dtype):
    """vitb200_attention_tc_lse then vitb200_attention_probs on random q / k / v against a float64 softmax of the same
    16-bit q / k; the attention output of the lse variant is the bits of vitb200_attention_tc's.  Scores spread over
    +-40 nats in some heads, so rows hold underflowing probabilities."""
    batch, heads = 3, 4
    tdt = torch.float16 if dtype == _lib.DT_F16 else torch.bfloat16
    g = torch.Generator().manual_seed(T + dtype)
    qkv = torch.randn((batch, T, 3, heads, 64), generator=g)
    qkv[:, :, :2] *= torch.tensor([0.5, 1.0, 2.0, 3.0]).view(1, 1, 1, heads, 1)      # head h: scores ~ (0.25 .. 9)^2
    qkv16 = qkv.reshape(batch * T, 3 * heads * 64).to(tdt).cuda()
    out_ref = torch.empty((batch * T, heads * 64), dtype=tdt, device="cuda")
    out = torch.empty_like(out_ref)
    lse = torch.empty((batch * heads, T), dtype=torch.float32, device="cuda")
    maps = torch.full((batch, heads, T, T), float("nan"), device="cuda")
    _lib.check(lib.vitb200_attention_tc(stream(), qkv16.data_ptr(), out_ref.data_ptr(), batch, T, heads, dtype))
    _lib.check(lib.vitb200_attention_tc_lse(stream(), qkv16.data_ptr(), out.data_ptr(), lse.data_ptr(), batch, T, heads, dtype))
    _lib.check(lib.vitb200_attention_probs(stream(), qkv16.data_ptr(), lse.data_ptr(), maps.data_ptr(), batch, T, heads, dtype))
    torch.cuda.synchronize()
    assert torch.equal(out, out_ref)
    q16 = qkv16.view(batch, T, 3, heads, 64).to(torch.float64).cpu()
    q, k = q16[:, :, 0].transpose(1, 2), q16[:, :, 1].transpose(1, 2)
    ref = torch.softmax((q @ k.transpose(-1, -2)) * 0.125, dim=-1).numpy()
    got = maps.cpu().numpy()
    assert np.isfinite(got).all() and got.min() >= 0 and got.max() <= 1       # every element written (NaN-filled before)
    # the scores are fp32 sums of exact products of 16-bit values: a few ulps of sum_d |q_d k_d| each; an element's
    # exponent carries its own score's error and the row log-sum-exp's (at most the row's largest), ex2.approx / lg2.approx
    # and the fp32 row sum of the forward a few 1e-7 more
    mag = (q.abs() @ k.abs().transpose(-1, -2)).numpy() * 0.125
    rel = 2.0 ** -20 * (mag + mag.max(-1, keepdims=True)) + 4e-6
    err = np.abs(got - ref)
    assert (err <= rel * ref + 1e-30).all(), f"max rel error {float((err / np.maximum(ref, 1e-30)).max()):.2e}"
    assert np.abs(got.sum(-1) - 1).max() < 1e-5
    zero = got == 0
    assert not zero.any() or float(ref[zero].max()) < 2.0 ** -120
    # the row log-sum-exp is that of the same scores
    s = (q @ k.transpose(-1, -2)).numpy() * 0.125 * np.log2(np.e)
    want_lse = np.log2(np.exp2(s - s.max(-1, keepdims=True)).sum(-1)) + s.max(-1)
    assert np.abs(lse.cpu().numpy().reshape(batch, heads, T) - want_lse).max() < 1e-4 * max(1.0, np.abs(want_lse).max())


@pytest.mark.parametrize("T", [197, 257])
def test_non_finite_queries_give_nan_rows_not_valid_looking_maps(lib, T):
    """A NaN in q (an overflowed to_qkv output, a diverged model) must not come out of the clamp at 1 as a plausible
    probability: that query's row is NaN, every other row keeps its bits."""
    batch, heads, dt = 2, 2, _lib.DT_F16
    g = torch.Generator().manual_seed(T)
    qkv = torch.randn((batch * T, 3 * heads * 64), generator=g).to(torch.float16).cuda()
    bad = qkv.clone()
    bad[T + 5, 64 + 3] = float("nan")              # image 1, token 5, head 1, one q feature
    out = torch.empty((batch * T, heads * 64), dtype=torch.float16, device="cuda")
    lse = torch.empty((batch * heads, T), device="cuda")
    maps = []
    for src in (qkv, bad):
        m = torch.empty((batch, heads, T, T), device="cuda")
        _lib.check(lib.vitb200_attention_tc_lse(stream(), src.data_ptr(), out.data_ptr(), lse.data_ptr(), batch, T, heads, dt))
        _lib.check(lib.vitb200_attention_probs(stream(), src.data_ptr(), lse.data_ptr(), m.data_ptr(), batch, T, heads, dt))
        maps.append(m)
    torch.cuda.synchronize()
    clean, got = maps
    assert bool(torch.isnan(got[1, 1, 5]).all())
    rest = torch.ones((batch, heads, T), dtype=torch.bool, device="cuda")
    rest[1, 1, 5] = False
    assert torch.equal(got[rest], clean[rest])


# ---------------------------------------------------------------- errors
def test_fp32_handle_is_unsupported_in_the_c_call(lib):
    cfg = TINY
    eng = Engine(**cfg, precision="fp32", max_batch=2)
    eng.load_params(perturb_params(init_params(seed=0, **cfg)))
    x = torch.zeros((2, 32, 32, 3), device="cuda")
    logits = torch.empty((2, 8), device="cuda")
    maps = torch.empty((2, 1, 2, 17, 17), device="cuda")
    layers = (C.c_int * 1)(0)
    rc = lib.vitb200_forward_attn(eng.handle, stream(), x.data_ptr(), 2, logits.data_ptr(), layers, 1, maps.data_ptr())
    assert rc == -4   # VITB200_ERR_UNSUPPORTED
    assert b"fp32" in lib.vitb200_last_error()
    with pytest.raises(ValueError, match="fp32"):
        eng.forward_attn(x, [0])
    eng.close()


def test_c_call_rejects_bad_layers(lib):
    cfg = TINY
    eng = Engine(**cfg, precision="fp16", max_batch=2)
    eng.load_params(perturb_params(init_params(seed=0, **cfg)))
    x = torch.zeros((2, 32, 32, 3), device="cuda")
    logits = torch.empty((2, 8), device="cuda")
    maps = torch.empty((2, 2, 2, 17, 17), device="cuda")
    for ls in ([0, 0], [0, 2], [-1, 1]):
        arr = (C.c_int * 2)(*ls)
        assert lib.vitb200_forward_attn(eng.handle, stream(), x.data_ptr(), 2, logits.data_ptr(), arr, 2, maps.data_ptr()) == -1
    arr = (C.c_int * 2)(0, 1)
    assert lib.vitb200_forward_attn(eng.handle, stream(), x.data_ptr(), 2, logits.data_ptr(), arr, 3, maps.data_ptr()) == -1
    assert lib.vitb200_forward_attn(eng.handle, stream(), x.data_ptr(), 2, logits.data_ptr(), arr, 2, None) == -1
    eng.close()


def test_python_errors_come_before_device_work(lib):
    cfg = TINY
    variables = perturb_params(init_params(seed=0, **cfg))
    x = torch.as_tensor(images_for(cfg, 2), device="cuda")
    v = ViT(**cfg)
    v.apply(variables, x)                       # engine built and loaded
    torch.cuda.synchronize()
    n0 = launch_count()
    for kw, match in (({"layers": [2]}, "outside"), ({"layers": [1, 1]}, "distinct"), ({"precision": "fp32"}, "fp32")):
        with pytest.raises(ValueError, match=match):
            v.attention_maps(variables, x, **kw)
    assert launch_count() == n0
    eng = Engine(**cfg, precision="fp16", max_batch=2)
    eng.load_params(variables)
    n0 = launch_count()
    for bad in (torch.empty((2, 1, 2, 17, 16), device="cuda"), torch.empty((2, 1, 2, 17, 17), device="cuda", dtype=torch.float16),
                torch.empty((2, 1, 2, 17, 17))):
        with pytest.raises(ValueError, match="maps must be"):
            eng.forward_attn(x, [0], maps=bad)
    assert launch_count() == n0
    eng.close()
