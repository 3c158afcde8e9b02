"""The on-device training step's host side, without a GPU: the float64 references the GPU tests use (AdamW against
torch.optim.AdamW, cross-entropy against torch autograd), mask parsing, and the checks that run before device work."""
import numpy as np
import pytest
import torch

from vit_flax_b200 import adamw
from vit_flax_b200.optim import parse_mask_tree
from vit_flax_b200.train import check_labels
from _adamw_oracle import adamw_ref, xent_ref

SHAPES = {"Dense_0/kernel": (6, 5), "Dense_0/bias": (5,), "LayerNorm_0/scale": (5,), "Dense_1/kernel": (5, 3)}


def test_adamw_ref_matches_torch_adamw_float64():
    """Four steps with weight decay, a decay mask (two param groups), clipping and a learning-rate schedule."""
    rng = np.random.default_rng(0)
    params = {k: rng.standard_normal(s) for k, s in SHAPES.items()}
    decay = {k: k.endswith("kernel") for k in SHAPES}
    tp = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params.items()}
    sched = lambda i: 1e-2 * (0.5 ** i)
    hp = dict(b1=0.8, b2=0.95, eps=1e-6, weight_decay=0.1)
    opt = torch.optim.AdamW([{"params": [tp[k] for k in SHAPES if decay[k]], "weight_decay": hp["weight_decay"]},
                             {"params": [tp[k] for k in SHAPES if not decay[k]], "weight_decay": 0.0}],
                            lr=sched(0), betas=(hp["b1"], hp["b2"]), eps=hp["eps"])
    mu = {k: np.zeros(s) for k, s in SHAPES.items()}
    nu = {k: np.zeros(s) for k, s in SHAPES.items()}
    count, max_norm, scale = 0, 3.0, 0.25
    for step in range(4):
        raw = {k: rng.standard_normal(s) * (4.0 if step % 2 else 0.5) for k, s in SHAPES.items()}
        params, mu, nu, count, skipped, norm = adamw_ref(params, raw, mu, nu, count, lr=sched(step), decay=decay,
                                                         max_grad_norm=max_norm, grad_scale=scale, **hp)
        assert skipped == 0 and count == step + 1
        g = {k: torch.tensor(raw[k] * scale) for k in SHAPES}
        tnorm = float(torch.sqrt(sum((v * v).sum() for v in g.values())))
        assert norm == pytest.approx(tnorm, rel=1e-12)
        for k in SHAPES:       # optax.clip_by_global_norm: g * max_norm / max(norm, max_norm)
            tp[k].grad = g[k] * (max_norm / max(tnorm, max_norm))
        for group in opt.param_groups:
            group["lr"] = sched(step)
        opt.step()
        for k in SHAPES:
            np.testing.assert_allclose(params[k], tp[k].detach().numpy(), rtol=1e-12, atol=1e-14)
            np.testing.assert_allclose(mu[k], opt.state[tp[k]]["exp_avg"].numpy(), rtol=1e-12, atol=1e-14)
            np.testing.assert_allclose(nu[k], opt.state[tp[k]]["exp_avg_sq"].numpy(), rtol=1e-12, atol=1e-14)


def test_adamw_ref_skips_non_finite_and_freezes():
    rng = np.random.default_rng(1)
    params = {k: rng.standard_normal(s) for k, s in SHAPES.items()}
    zeros = {k: np.zeros(s) for k, s in SHAPES.items()}
    g = {k: rng.standard_normal(s) for k, s in SHAPES.items()}
    g["Dense_0/bias"][2] = np.inf
    p2, m2, n2, count, skipped, _ = adamw_ref(params, g, zeros, zeros, 5, lr=1e-2)
    assert skipped == 1 and count == 5
    assert all(np.array_equal(p2[k], params[k]) and not m2[k].any() for k in SHAPES)
    trainable = {k: k != "Dense_0/bias" for k in SHAPES}   # the only non-finite leaf is frozen: the step applies
    p2, _, _, count, skipped, _ = adamw_ref(params, g, zeros, zeros, 5, lr=1e-2, trainable=trainable)
    assert skipped == 0 and count == 6
    assert np.array_equal(p2["Dense_0/bias"], params["Dense_0/bias"])
    assert not np.array_equal(p2["Dense_0/kernel"], params["Dense_0/kernel"])


@pytest.mark.parametrize("eps", [0.0, 0.1])
@pytest.mark.parametrize("B,C", [(1, 10), (7, 37), (16, 1000)])
def test_xent_ref_matches_torch_cross_entropy(B, C, eps):
    rng = np.random.default_rng(B * C)
    z = rng.standard_normal((B, C)) * 3
    z[0, :3] = [1e4, -1e4, 5e3] if C >= 3 else z[0, :3]
    y = rng.integers(0, C, B)
    zt = torch.tensor(z, requires_grad=True)
    loss = torch.nn.functional.cross_entropy(zt, torch.tensor(y), label_smoothing=eps)
    loss.backward()
    got, dl = xent_ref(z, y, eps, dscale=4.0)
    assert got == pytest.approx(float(loss.detach()), rel=1e-12)
    np.testing.assert_allclose(dl, 4.0 * zt.grad.numpy(), rtol=1e-10, atol=1e-15)


def test_mask_forms():
    tx = adamw(1e-3, mask=lambda path, shape: len(shape) > 1)
    assert tx.decay_mask(SHAPES) == {k: len(s) > 1 for k, s in SHAPES.items()}
    assert adamw(1e-3).decay_mask(SHAPES) == {k: True for k in SHAPES}
    tree = {"Dense_0": {"kernel": True, "bias": False}, "LayerNorm_0": {"scale": np.bool_(False)}, "Dense_1": {"kernel": True}}
    want = {"Dense_0/kernel": True, "Dense_0/bias": False, "LayerNorm_0/scale": False, "Dense_1/kernel": True}
    assert adamw(1e-3, mask=tree).decay_mask(SHAPES) == want
    assert parse_mask_tree({"params": tree}, SHAPES) == want
    with pytest.raises(ValueError, match="missing"):
        parse_mask_tree({"Dense_0": {"kernel": True}}, SHAPES)
    with pytest.raises(ValueError, match="bool"):
        parse_mask_tree(dict(tree, Dense_1={"kernel": 1.0}), SHAPES)
    with pytest.raises(ValueError, match="mask"):
        adamw(1e-3, mask=[True])


def test_schedule_is_evaluated_per_step():
    tx = adamw(lambda i: 0.1 / (i + 1))
    assert tx.lr(0) == pytest.approx(0.1) and tx.lr(4) == pytest.approx(0.02)
    with pytest.raises(ValueError):
        adamw(lambda i: -1.0).lr(0)


@pytest.mark.parametrize("kw", [dict(learning_rate=-1.0), dict(learning_rate=float("nan")), dict(learning_rate="1e-3"),
                                dict(learning_rate=1e-3, b1=1.0), dict(learning_rate=1e-3, b2=-0.1),
                                dict(learning_rate=1e-3, eps=-1e-8), dict(learning_rate=1e-3, weight_decay=-0.1),
                                dict(learning_rate=1e-3, max_grad_norm=0.0), dict(learning_rate=1e-3, max_grad_norm=float("inf"))])
def test_bad_hyperparameters_raise(kw):
    with pytest.raises(ValueError):
        adamw(**kw)


def test_labels_are_checked_on_the_host():
    assert check_labels(np.array([0, 3, 1]), 3).dtype == torch.int32
    assert check_labels(torch.tensor([2, 1], dtype=torch.int64), 2).dtype == torch.int64
    for bad in (np.array([0.0, 1.0, 2.0]), np.array([[0], [1], [2]]), np.array([0, 1]), torch.tensor([0.5, 1.0, 2.0]),
                torch.tensor([True, False, True]), ["a", "b", "c"]):
        with pytest.raises(ValueError):
            check_labels(bad, 3)
