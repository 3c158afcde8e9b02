"""The class-token tail of the forward on a real B200 (DESIGN.md section 3).

With pool='cls' and no dropout the last block computes attention for q tile 0 alone and runs to_out / FeedForward over
the B class-token rows.  A forward that records the last layer's attention weights runs that block in full, so
``attention_maps(..., layers=[depth - 1])`` is the reference the pruned logits must equal bit for bit; both are also
held to the CPU oracle as the full forward is (tests/test_gpu_forward.py)."""
import numpy as np
import pytest
import torch

from oracle import vit_torch
from vit_flax_b200 import ViT, init_params, perturb_params
from vit_flax_b200._lib import VitB200Error
from vit_flax_b200.engine import Engine, launch_count
from vit_flax_b200.runtime import clear_cache
from _util import C2, C4, C5, images_for

pytestmark = pytest.mark.gpu

C1_GEOM = dict(image_size=128, patch_size=16, num_classes=10, dim=256, depth=2, heads=4, mlp_dim=512)   # T = 65
GEOMETRIES = {
    "t65": C1_GEOM,                       # one key block of 64 + 1: a 65-row q tile, tile modes of small GEMMs
    "t197": dict(C2, depth=2),            # ViT-B/16: 2 q tiles, attention_tc5
    "t257": dict(C4, depth=2),            # ViT-H/14: 3 q tiles, attention_tc5m (two key blocks)
    "t1025": dict(C5, depth=2),           # 512-px ViT-L/16: 9 q tiles, attention_tc5m (six key blocks)
}
# batches, largest first so one engine serves them all: 300 leaves a ragged 128-row block of class rows (300 = 2 x 128 + 44),
# 41 x 197 token rows still take the captured-graph path (<= 8192), 42 x 197 no longer do
BATCHES = {"t65": [300, 42, 41, 1], "t197": [300, 42, 41, 2, 1], "t257": [42, 41, 2], "t1025": [3, 1]}
TOL = {"fp16": 2e-2, "bf16": 2e-2}


@pytest.fixture(autouse=True)
def _fresh_cache():
    yield
    clear_cache()
    torch.cuda.empty_cache()


def _model(cfg, seed=1):
    return perturb_params(init_params(seed=seed, **cfg), seed=seed + 1)


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("geom", list(GEOMETRIES))
def test_pruned_logits_equal_the_full_last_block(geom, precision):
    cfg = GEOMETRIES[geom]
    v = ViT(**cfg)
    variables = _model(cfg)
    last = cfg["depth"] - 1
    for batch in BATCHES[geom]:
        x = torch.as_tensor(images_for(cfg, batch, seed=batch), device="cuda")
        pruned = v.apply(variables, x, precision=precision)
        full, _ = v.attention_maps(variables, x, layers=[last], precision=precision)
        torch.cuda.synchronize()
        assert bool(torch.isfinite(pruned).all())
        diff = float((pruned - full).abs().max())
        assert torch.equal(pruned, full), f"{geom} {precision} batch {batch}: max |pruned - full| {diff:.3e}"


def test_launch_count_is_unchanged():
    """The tail keeps the schedule's launches: 4 + 5L with the LayerNorm fold, 4 + 7L on the LayerNorm-kernel schedule."""
    cfg = GEOMETRIES["t197"]
    variables = _model(cfg)
    x = torch.as_tensor(images_for(cfg, 42, seed=3), device="cuda")
    for precision, per_layer in (("fp16", 5), ("fp8", 7)):
        v = ViT(**cfg)
        v.apply(variables, x, precision=precision)
        torch.cuda.synchronize()
        n0 = launch_count()
        v.apply(variables, x, precision=precision)
        assert launch_count() - n0 == 4 + per_layer * cfg["depth"], precision


def _oracle(variables, img, cfg, pool="cls", operand_dtype=None, ln_fold=True):
    return vit_torch.vit_forward(vit_torch.tree_to_torch(variables), img, pool=pool, operand_dtype=operand_dtype,
                                 ln_fold=ln_fold, **cfg).numpy()


def _bound(precision, variables, img, cfg, want, pool="cls"):
    if precision == "fp16":
        return TOL["fp16"]
    emu = _oracle(variables, img, cfg, pool, torch.bfloat16)
    return max(TOL["bf16"], 1.25 * float(np.abs(emu - want).max()))   # tests/test_gpu_forward.py: bf16_bound


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("geom", list(GEOMETRIES))
def test_pruned_logits_against_the_oracle(geom, precision):
    cfg = GEOMETRIES[geom]
    variables = _model(cfg, seed=5)
    img = images_for(cfg, 2, seed=7)
    want = _oracle(variables, img, cfg)
    got = ViT(**cfg).apply(variables, img, precision=precision)
    err = float(np.abs(got - want).max())
    tol = _bound(precision, variables, img, cfg, want)
    print(f"[cls tail] {geom} {precision}: max abs logit error {err:.2e} (bound {tol:.2e})")
    assert err < tol


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_mean_pooling_keeps_the_full_forward(precision):
    cfg = GEOMETRIES["t197"]
    variables = _model(cfg, seed=9)
    img = images_for(cfg, 2, seed=11)
    v = ViT(pool="mean", **cfg)
    want = _oracle(variables, img, cfg, pool="mean")
    got = v.apply(variables, img, precision=precision)
    err = float(np.abs(got - want).max())
    tol = _bound(precision, variables, img, cfg, want, pool="mean")
    assert err < tol, f"mean pool {precision}: {err:.3e} > {tol:.3e}"
    eng = Engine(**cfg, pool="mean", precision=precision, max_batch=2)
    eng.load_params(variables)
    eng.forward_host(img)
    tok = eng.tokens_after_transformer(2)          # every row is computed: readable
    assert tok.shape == (2, 197, cfg["dim"]) and np.isfinite(tok).all()
    eng.close()


@pytest.mark.parametrize("batch", [42, 2])
def test_fp8_pruned_logits_equal_the_full_last_block(batch):
    cfg = GEOMETRIES["t197"]
    v = ViT(**cfg)
    variables = _model(cfg, seed=13)
    x = torch.as_tensor(images_for(cfg, batch, seed=15), device="cuda")
    pruned = v.apply(variables, x, precision="fp8")
    full, _ = v.attention_maps(variables, x, layers=[cfg["depth"] - 1], precision="fp8")
    torch.cuda.synchronize()
    assert torch.equal(pruned, full), f"fp8 batch {batch}: max |pruned - full| {float((pruned - full).abs().max()):.3e}"


@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp8"])
def test_tokens_after_a_pruned_forward(precision):
    """The token stream is incomplete after a pruned forward: reading it raises instead of returning stale rows; a forward
    that records the last layer runs it in full, and its class rows are the ones the pruned forward pooled."""
    cfg = GEOMETRIES["t65"]
    variables = _model(cfg, seed=17)
    img = images_for(cfg, 3, seed=19)
    eng = Engine(**cfg, precision=precision, max_batch=3)
    eng.load_params(variables)
    x = torch.as_tensor(img, device="cuda")
    pruned = eng.forward(x)
    with pytest.raises(VitB200Error, match="class-token"):
        eng.tokens_after_transformer(3)
    full, _ = eng.forward_attn(x, [cfg["depth"] - 1])
    tok = eng.tokens_after_transformer(3)
    assert tok.shape == (3, 65, cfg["dim"]) and np.isfinite(tok).all()
    assert torch.equal(pruned, full)
    # a recording forward of another layer prunes again
    eng.forward_attn(x, [0])
    with pytest.raises(VitB200Error):
        eng.tokens_after_transformer(3)
    eng.close()


def test_dropout_keeps_the_full_forward():
    """Dropout masks are indexed by token row: a forward with rates > 0 runs the whole last block."""
    cfg = GEOMETRIES["t65"]
    eng = Engine(**cfg, precision="fp16", max_batch=2, dropout=0.1)
    eng.load_params(_model(cfg, seed=21))
    eng.set_dropout_key(7)
    eng.forward_host(images_for(cfg, 2, seed=23))
    tok = eng.tokens_after_transformer(2)
    assert np.isfinite(tok).all()
    eng.close()
