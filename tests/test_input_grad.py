"""Gradients with respect to the input images, the parts that need no GPU: the float64 checker of
``tests/_input_grad_oracle.py`` against central differences of the oracle's forward, the argument checks of
``vjp(wrt=...)`` and the C ABI declarations."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import vit_torch
from vit_flax_b200 import SimpleViT, ViT, _lib, init_params, perturb_params
from vit_flax_b200.params import flatten_params
from _input_grad_oracle import vit_vjp_images
from _util import TINY, TINY_MEAN, images_for

HEADER = Path(__file__).resolve().parents[1] / "include" / "vitb200.h"


def _forward64(variables, img, **cfg):
    return vit_torch.vit_forward(vit_torch.tree_to_torch(variables, torch.float64), img, **cfg).numpy()


@pytest.mark.parametrize("cfg,pool,drop", [(TINY, "cls", 0.0), (TINY_MEAN, "mean", 0.0), (TINY, "cls", 0.1),
                                           (TINY_MEAN, "mean", 0.1)])
def test_oracle_image_gradient_matches_central_differences(cfg, pool, drop):
    """dL/dx of the float64 autograd checker at 20 sampled pixels against central differences of the forward, with
    the dropout masks (rate 0.1 everywhere, one fixed key) held fixed like the backward pass replays them."""
    kw = dict(cfg, pool=pool)
    if drop:
        kw.update(dropout=drop, emb_dropout=drop, dropout_key=0x1234)
    variables = perturb_params(init_params(seed=5, **cfg), seed=6)
    img = images_for(cfg, 2, seed=7).astype(np.float64)
    dl = np.random.default_rng(8).standard_normal((2, cfg["num_classes"]))
    _, _, dx = vit_vjp_images(variables, img, dl, **kw)
    assert dx.shape == img.shape and np.abs(dx).max() > 0
    rng = np.random.default_rng(9)
    idx = [tuple(int(rng.integers(0, s)) for s in img.shape) for _ in range(20)]
    eps = 1e-5
    got, fd = [], []
    for i in idx:
        vals = []
        for sgn in (1, -1):
            x = img.copy()
            x[i] += sgn * eps
            vals.append(float((_forward64(variables, x, **kw) * dl).sum()))
        fd.append((vals[0] - vals[1]) / (2 * eps))
        got.append(dx[i])
    got, fd = np.array(got), np.array(fd)
    assert np.abs(got - fd).max() / np.abs(got).max() <= 1e-6, (got, fd)


@pytest.mark.parametrize("pool", ["cls", "mean"])
def test_asking_for_the_image_gradient_leaves_the_parameter_gradients_unchanged(pool):
    variables = perturb_params(init_params(seed=11, **TINY), seed=12)
    img = images_for(TINY, 3, seed=13)
    dl = np.random.default_rng(14).standard_normal((3, TINY["num_classes"]))
    logits_a, ga = vit_torch.vit_vjp(variables, img, dl, pool=pool, **TINY)
    logits_b, gb, _ = vit_vjp_images(variables, img, dl, pool=pool, **TINY)
    np.testing.assert_array_equal(logits_a, logits_b)
    fa, fb = flatten_params({"params": ga}), flatten_params({"params": gb})
    assert set(fa) == set(fb)
    for k in fa:
        np.testing.assert_array_equal(fa[k], fb[k], err_msg=k)


def test_unknown_wrt_is_rejected_before_any_device_work():
    img = images_for(TINY, 1)
    with pytest.raises(ValueError, match="wrt"):
        ViT(**TINY).vjp({}, img, wrt="bogus")
    with pytest.raises(ValueError, match="wrt"):
        ViT(**TINY).vjp({}, img, wrt="images")
    with pytest.raises(ValueError, match="wrt"):
        SimpleViT(image_size=32, patch_size=8, num_classes=4, dim=64, depth=1, heads=1, mlp_dim=64).vjp(
            {}, np.zeros((1, 3, 32, 32), np.float32), wrt=None)


def test_gradient_flags_match_the_header():
    text = HEADER.read_text()
    flags = dict(re.findall(r"#define (VITB200_GRAD_\w+)\s+(\d+)", text))
    assert flags == {"VITB200_GRAD_PARAMS": str(_lib.GRAD_PARAMS), "VITB200_GRAD_IMAGES": str(_lib.GRAD_IMAGES)}
    assert "vitb200_backward_ex" in _lib.SIGNATURES and "vitb200_unpatchify" in _lib.SIGNATURES
