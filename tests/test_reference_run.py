"""The oracle (and on a GPU the CUDA path) against OUTPUTS OF THE REFERENCE ITSELF.

tests/golden/ref_vit.npz and ref_simple_vit.npz were written by tests/golden/make_reference_golden.py, which executes
the reference's vit_flax/vit.py and simple_vit.py unmodified over oracle/flax_shim (a numpy restatement of the jax /
flax API they use; its README states what that pins and what it does not).  Where VIT_FLAX_REFERENCE names the
reference's vit_flax/ directory, the reference is also re-run live and compared with the committed fixtures.
"""
import importlib.util
import sys
from pathlib import Path

import numpy as np
import pytest

from _util import C1, GOLDEN, TINY, TINY_MEAN, load_golden

ROOT = Path(__file__).resolve().parents[1]
spec = importlib.util.spec_from_file_location("make_reference_golden", GOLDEN / "make_reference_golden.py")
mrg = importlib.util.module_from_spec(spec)
spec.loader.exec_module(mrg)

from oracle import simple_vit_numpy, vit_numpy, vit_torch  # noqa: E402
from vit_flax_b200 import ViT, init_params, perturb_params  # noqa: E402
from vit_flax_b200.params import count_params, flatten_params  # noqa: E402
from vit_flax_b200.simple_vit import SimpleViT  # noqa: E402


@pytest.fixture(scope="module")
def ref_vit():
    return np.load(GOLDEN / "ref_vit.npz")


@pytest.fixture(scope="module")
def ref_simple():
    return np.load(GOLDEN / "ref_simple_vit.npz")


def simple_tree(ref_simple):
    tree = {}
    for k in ref_simple.files:
        if not k.startswith("param."):
            continue
        node = tree
        parts = k[len("param."):].split(".")
        for p in parts[:-1]:
            node = node.setdefault(p, {})
        node[parts[-1]] = ref_simple[k]
    return {"params": tree}


def c1_inputs():
    return (perturb_params(init_params(seed=1, **C1), seed=2),
            np.random.default_rng(0).standard_normal((1, 256, 256, 3)).astype(np.float32))


# ------------------------------------------------------------------ oracle vs the reference run (CPU)
def test_numpy_oracle_reproduces_the_reference_run(ref_vit):
    variables, meta = load_golden("tiny_cls.npz")
    y = vit_numpy.vit_forward(variables, meta["images"], **TINY)
    assert np.abs(y - ref_vit["tiny_cls_logits"]).max() < 1e-10
    variables, meta = load_golden("tiny_mean.npz")
    y = vit_numpy.vit_forward(variables, meta["images"], pool="mean", **TINY_MEAN)
    assert np.abs(y - ref_vit["tiny_mean_logits"]).max() < 1e-10
    variables, img = c1_inputs()
    y = vit_numpy.vit_forward(variables, img, **C1)
    assert y.shape == (1, 1000) and np.abs(y - ref_vit["c1_logits"]).max() < 1e-9


def test_oracle_written_fixtures_equal_the_reference_run(ref_vit):
    """tiny_cls / tiny_mean / c1_logits.npz were written from the oracle in round 1; the reference computes the same."""
    for name, key in (("tiny_cls.npz", "tiny_cls_logits"), ("tiny_mean.npz", "tiny_mean_logits"), ("c1_logits.npz", "c1_logits")):
        _, meta = load_golden(name)
        assert np.abs(meta["logits"] - ref_vit[key]).max() < 1e-9, name


def test_torch_oracle_reproduces_the_reference_run(ref_vit):
    variables, meta = load_golden("tiny_cls.npz")
    y = vit_torch.vit_forward(vit_torch.tree_to_torch(variables), meta["images"], **TINY).numpy()
    assert np.abs(y - ref_vit["tiny_cls_logits"]).max() < 2e-5
    variables, img = c1_inputs()
    y = vit_torch.vit_forward(vit_torch.tree_to_torch(variables), img, **C1).numpy()
    assert np.abs(y - ref_vit["c1_logits"]).max() < 1e-4


def test_dropped_forward_matches_the_reference_run(ref_vit):
    """dropout = emb_dropout = 0.1 (README usage): the reference, handed the masks of oracle/philox.py in its own
    Dropout call order, and the oracle's site numbering (0 embedding, then per layer to_out / gelu / FF output) agree; the
    only difference is the keep scale, float32(1 / 0.9) in the oracle as in the kernels."""
    variables, meta = load_golden("tiny_cls.npz")
    y = vit_numpy.vit_forward(variables, meta["images"], dropout=0.1, emb_dropout=0.1,
                              dropout_key=int(ref_vit["dropout_key"]), **TINY)
    assert np.abs(y - ref_vit["tiny_cls_dropout_logits"]).max() < 1e-6
    assert np.abs(ref_vit["tiny_cls_dropout_logits"] - ref_vit["tiny_cls_logits"]).max() > 1e-2   # the masks did act
    assert bool(ref_vit["dropout_without_rng_raises"])      # deterministic=False: a rate > 0 needs the 'dropout' rng


def test_init_pytree_is_the_one_the_reference_constructs(ref_vit, ref_simple):
    """Leaf names and shapes of the reference's own `init` (its module construction order under Flax's compact
    auto-naming) == the tree `vit_flax_b200.ViT.init` / `SimpleViT.init` emit and the engine looks leaves up by."""
    want = dict(zip(ref_vit["init_names"].tolist(), ref_vit["init_shapes"].tolist()))
    got = {k: ",".join(map(str, np.shape(v))) for k, v in
           flatten_params(ViT(**TINY).init({"params": 0}, np.zeros((1, 32, 32, 3), np.float32))).items()}
    assert got == want
    want = dict(zip(ref_simple["init_names"].tolist(), ref_simple["init_shapes"].tolist()))
    got = {k: ",".join(map(str, np.shape(v))) for k, v in
           flatten_params(SimpleViT(**mrg.SIMPLE_TINY).init({"params": 0}, np.zeros((1, 3, 32, 32), np.float32))).items()}
    assert got == want
    assert {"LayerNorm_0/scale", "Dense_0/kernel", "Dense_1/kernel"} <= set(want)         # head = Dense_0, patch = Dense_1
    assert want["Dense_1/kernel"] == "192,64" and want["Dense_0/kernel"] == "64,10"


def test_reference_demo_blocks(ref_vit, ref_simple):
    """`python vit.py` / `python simple_vit.py`: output shape and parameter count as the reference prints them."""
    assert ref_vit["demo_stdout"].tolist() == ["(1, 1000)", "Number of parameters in Flax model: 54622184"]
    assert count_params(**C1) == 54622184
    assert ref_simple["demo_stdout"].tolist() == ["(1, 1000)", "Number of parameters in Flax model: 54535144"]
    demo = dict(image_size=256, patch_size=32, num_classes=1000, dim=1024, depth=6, heads=16, mlp_dim=2048)
    tree = SimpleViT(**demo).init({"params": 0}, np.zeros((1, 3, 256, 256), np.float32))
    assert sum(int(np.prod(np.shape(v))) for v in flatten_params(tree).values()) == 54535144


def test_simple_vit_oracle_reproduces_the_reference_run(ref_simple):
    y = simple_vit_numpy.simple_vit_forward(simple_tree(ref_simple), ref_simple["images"], **mrg.SIMPLE_TINY)
    assert np.abs(y - ref_simple["logits"]).max() < 1e-10


@pytest.mark.skipif(not mrg.reference_available(),
                    reason="needs the reference's sources: set VIT_FLAX_REFERENCE to a vit-flax checkout's vit_flax/ directory")
def test_fixtures_are_what_the_reference_computes_today(ref_vit, ref_simple):
    vit_out, simple_out = mrg.generate()
    for want, got in ((ref_vit, vit_out), (ref_simple, simple_out)):
        assert sorted(want.files) == sorted(got)
        for k in want.files:
            a, b = want[k], np.asarray(got[k])
            if a.dtype.kind in "fc":
                assert np.abs(a - b).max() < 1e-12, k
            else:
                assert (a == b).all(), k


# ------------------------------------------------------------------ the shim's own rules (CPU)
def test_shim_naming_and_scope_rules():
    with mrg.shimmed():
        import flax.linen as nn
        import jax

        class Inner(nn.Module):
            @nn.compact
            def __call__(self, x):
                return nn.Dense(3)(x)

        class Holder(nn.Module):
            fn: object

            @nn.compact
            def __call__(self, x):
                return self.fn(x) + nn.Dense(3)(x)

        class Outer(nn.Module):
            @nn.compact
            def __call__(self, x):
                a, b = Holder(Inner()), Holder(Inner())
                return a(x) + b(x)

        x = np.ones((2, 4))
        tree = Outer().init(jax.random.PRNGKey(0), x)["params"]
        # Inner is constructed in Outer's scope -> Outer's child, not Holder's (flax adopts only parent-less modules)
        assert sorted(tree) == ["Holder_0", "Holder_1", "Inner_0", "Inner_1"]
        assert sorted(tree["Holder_0"]) == ["Dense_0"] and sorted(tree["Inner_1"]) == ["Dense_0"]
        y = Outer().apply({"params": tree}, x)
        assert y.shape == (2, 3)
        bad = {"Holder_0": tree["Holder_0"], "Holder_1": tree["Holder_1"], "Inner_0": tree["Inner_0"]}
        with pytest.raises(KeyError):
            Outer().apply({"params": bad}, x)
        with pytest.raises(ValueError):
            Outer().apply({"params": tree}, np.ones((2, 5)))          # kernel shape check
        with pytest.raises(RuntimeError):
            Outer()(x)                                                  # unbound module
        with pytest.raises(ValueError):
            nn.Dropout(0.5).apply({}, x, deterministic=False)          # needs the 'dropout' rng
        assert nn.Dropout(0.0).apply({}, x, deterministic=False) is x
    assert "flax" not in sys.modules and "jax" not in sys.modules


# ------------------------------------------------------------------ the CUDA path vs the reference run (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("fp16", 2e-2)])
def test_gpu_forward_matches_the_reference_run(ref_vit, precision, tol):
    variables, meta = load_golden("tiny_cls.npz")
    y = ViT(**TINY).apply(variables, meta["images"], precision=precision)
    assert np.abs(y - ref_vit["tiny_cls_logits"]).max() < tol
    variables, meta = load_golden("tiny_mean.npz")
    y = ViT(pool="mean", **TINY_MEAN).apply(variables, meta["images"], precision=precision)
    assert np.abs(y - ref_vit["tiny_mean_logits"]).max() < tol
    variables, img = c1_inputs()
    y = ViT(**C1).apply(variables, img, precision=precision)
    assert y.shape == (1, 1000) and np.abs(y - ref_vit["c1_logits"]).max() < tol


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("fp16", 2e-2)])
def test_gpu_dropped_forward_matches_the_reference_run(ref_vit, precision, tol):
    variables, meta = load_golden("tiny_cls.npz")
    y = ViT(dropout=0.1, emb_dropout=0.1, **TINY).apply(variables, meta["images"], precision=precision,
                                                         rngs={"dropout": int(ref_vit["dropout_key"])})
    assert np.abs(y - ref_vit["tiny_cls_dropout_logits"]).max() < tol


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("fp16", 2e-2)])
def test_gpu_simple_vit_matches_the_reference_run(ref_simple, precision, tol):
    y = SimpleViT(**mrg.SIMPLE_TINY).apply(simple_tree(ref_simple), ref_simple["images"], precision=precision)
    assert np.abs(y - ref_simple["logits"]).max() < tol
