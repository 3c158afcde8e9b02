"""Attention maps without a GPU: the checker in tests/_attn_oracle.py against the torch oracle, the error floor of the
16-bit formats that sets the GPU tolerance, and every argument error of ``attention_maps`` raised before device work."""
import numpy as np
import pytest
import torch

from oracle import vit_numpy, vit_torch
from vit_flax_b200 import SimpleViT, ViT
from vit_flax_b200.engine import check_layers, check_maps
from _attn_oracle import error_floor, simple_vit_attention_maps, vit_attention_maps
from _util import TINY, TINY_MEAN, load_golden

GOLDEN = [("tiny_cls.npz", TINY), ("tiny_mean.npz", dict(TINY_MEAN, pool="mean"))]


def torch_oracle_maps(variables, images, cfg, monkeypatch):
    """Every layer's softmax(q k^T * 64^-0.5) from ``oracle.vit_torch`` at float64 (its attention goes through
    scaled_dot_product_attention, which is replaced here by the explicit softmax it computes)."""
    rec = []

    def sdpa(q, k, v, *a, **kw):
        att = torch.softmax((q @ k.transpose(-1, -2)) * q.shape[-1] ** -0.5, dim=-1)
        rec.append(att)
        return att @ v

    monkeypatch.setattr(torch.nn.functional, "scaled_dot_product_attention", sdpa)
    logits = vit_torch.vit_forward(vit_torch.tree_to_torch(variables, torch.float64), images, **cfg)
    return logits.numpy(), torch.stack(rec, dim=1).numpy()


@pytest.mark.parametrize("name,cfg", GOLDEN)
def test_oracle_maps_match_the_torch_oracle(name, cfg, monkeypatch):
    variables, meta = load_golden(name)
    logits, maps = vit_attention_maps(variables, meta["images"], **cfg)
    t_logits, t_maps = torch_oracle_maps(variables, meta["images"], cfg, monkeypatch)
    b, T = meta["images"].shape[0], maps.shape[-1]
    assert maps.shape == (b, cfg["depth"], cfg["heads"], T, T) and maps.dtype == np.float64
    np.testing.assert_allclose(maps, t_maps, rtol=0, atol=1e-12)
    np.testing.assert_allclose(logits, vit_numpy.vit_forward(variables, meta["images"], **cfg), rtol=0, atol=1e-12)
    np.testing.assert_allclose(logits, t_logits, rtol=0, atol=1e-10)
    assert np.abs(maps.sum(-1) - 1).max() < 1e-12 and maps.min() > 0
    # a subset in the order asked for is the same slices
    _, sub = vit_attention_maps(variables, meta["images"], layers=[cfg["depth"] - 1, 0], **cfg)
    np.testing.assert_array_equal(sub, maps[:, [cfg["depth"] - 1, 0]])


def test_oracle_maps_with_dropout_are_those_of_the_dropped_forward():
    """Dropout moves the residual stream (so the maps of later layers), never the weights themselves."""
    cfg = dict(TINY, depth=2)
    variables, meta = load_golden("tiny_cls.npz")
    key = 0xC0FFEE
    logits, maps = vit_attention_maps(variables, meta["images"], dropout=0.1, emb_dropout=0.2, dropout_key=key, **cfg)
    want = vit_numpy.vit_forward(variables, meta["images"], dropout=0.1, emb_dropout=0.2, dropout_key=key, **cfg)
    np.testing.assert_allclose(logits, want, rtol=0, atol=1e-12)
    _, plain = vit_attention_maps(variables, meta["images"], **cfg)
    assert np.abs(maps - plain).max() > 1e-3
    assert np.abs(maps.sum(-1) - 1).max() < 1e-12


def test_simple_vit_oracle_maps():
    from oracle import simple_vit_numpy
    cfg = dict(image_size=32, patch_size=8, num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128)
    v = SimpleViT(**cfg)
    img = np.random.default_rng(0).standard_normal((2, 3, 32, 32)).astype(np.float32)
    variables = v.init(0, img)
    logits, maps = simple_vit_attention_maps(variables, img, **cfg)
    assert maps.shape == (2, 2, 2, 16, 16)
    np.testing.assert_allclose(logits, simple_vit_numpy.simple_vit_forward(variables, img, **cfg), rtol=0, atol=1e-12)
    assert np.abs(maps.sum(-1) - 1).max() < 1e-12


@pytest.mark.parametrize("name,cfg", GOLDEN)
def test_error_floor_of_the_16_bit_formats(name, cfg):
    """The emulation's distance to the exact maps is the floor the GPU tolerance is built on (tests/_attn_oracle.py):
    pinned here so that a change of the emulation cannot silently widen it.  fp16 (11 significant bits) sits at a few
    1e-4, bf16 (8 bits) about eight times higher."""
    variables, meta = load_golden(name)
    _, exact = vit_attention_maps(variables, meta["images"], **cfg)
    f16 = error_floor(vit_attention_maps(variables, meta["images"], rounding="fp16", **cfg)[1], exact)
    bf16 = error_floor(vit_attention_maps(variables, meta["images"], rounding="bf16", **cfg)[1], exact)
    print(f"[attention maps] {name}: error floor fp16 {f16:.2e}, bf16 {bf16:.2e}")
    assert 1e-4 < f16 < 1e-3
    assert 1e-3 < bf16 < 1e-2
    assert 3 < bf16 / f16 < 20


@pytest.mark.parametrize("layers,match", [
    ([], "at least one"), ([0, 0], "distinct"), ([2], "outside"), ([-1], "outside"), ([0.5], "ints"),
    ([True], "ints"), (1, "sequence"), ("0", "sequence")])
def test_bad_layers_are_value_errors_before_device_work(layers, match):
    variables, meta = load_golden("tiny_cls.npz")
    with pytest.raises(ValueError, match=match):
        ViT(**TINY).attention_maps(variables, meta["images"], layers=layers)
    with pytest.raises(ValueError, match=match):
        check_layers(layers, TINY["depth"])
    img = np.zeros((1, 3, 32, 32), np.float32)
    with pytest.raises(ValueError, match=match):
        SimpleViT(image_size=32, patch_size=8, num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128).attention_maps(
            {}, img, layers=layers)


def test_layers_default_and_order():
    assert check_layers(None, 3) == [0, 1, 2]
    assert check_layers([2, np.int64(0)], 3) == [2, 0]


def test_fp32_precision_and_missing_dropout_key_are_value_errors():
    variables, meta = load_golden("tiny_cls.npz")
    with pytest.raises(ValueError, match="fp32"):
        ViT(**TINY).attention_maps(variables, meta["images"], precision="fp32")
    with pytest.raises(ValueError, match="fp32"):
        SimpleViT(image_size=32, patch_size=8, num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128).attention_maps(
            {}, np.zeros((1, 3, 32, 32), np.float32), precision="fp32")
    with pytest.raises(ValueError, match="rngs"):
        ViT(dropout=0.1, **TINY).attention_maps(variables, meta["images"])


@pytest.mark.parametrize("bad", ["shape", "dtype", "device", "layout", "type"])
def test_bad_maps_buffer_is_a_value_error(bad):
    """``Engine.forward_attn`` checks a caller's buffer with ``check_maps`` before it launches anything."""
    shape = (2, 1, 2, 17, 17)
    cpu = torch.device("cpu")
    maps, want_device = {
        "shape": (torch.empty((2, 1, 2, 17, 16)), cpu),
        "dtype": (torch.empty(shape, dtype=torch.float16), cpu),
        "device": (torch.empty(shape), torch.device("cuda", 0)),
        "layout": (torch.empty(shape).transpose(3, 4), cpu),
        "type": (np.empty(shape, np.float32), cpu)}[bad]
    with pytest.raises(ValueError, match="maps must be"):
        check_maps(torch, maps, shape, want_device)
    check_maps(torch, torch.empty(shape), shape, cpu)   # the right buffer passes
