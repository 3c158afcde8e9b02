"""Run the REFERENCE ITSELF and store what it computes:
    VIT_FLAX_REFERENCE=<checkout of conceptofmind/vit-flax>/vit_flax python tests/golden/make_reference_golden.py

Imports $VIT_FLAX_REFERENCE/vit.py and simple_vit.py UNMODIFIED (importlib, straight from where they lie) with
oracle/flax_shim on sys.path in place of the absent jax / flax (oracle/flax_shim/README.md says exactly what that shim
restates), runs their `init` / `apply` and their `__main__` demo blocks, and writes

    tests/golden/ref_vit.npz         logits of vit.py on the inputs + parameters of tiny_cls.npz / tiny_mean.npz /
                                     c1_logits.npz, the dropped forward (dropout = emb_dropout = 0.1), the token stream,
                                     the leaf names and shapes of `ViT.init`, the demo block's printed lines
    tests/golden/ref_simple_vit.npz  the same for simple_vit.py: init names / shapes, inputs, parameters and logits

The reference is not part of this repository; the fixtures are (tests/test_reference_run.py compares the oracle, and on
a GPU the CUDA path, with them; when VIT_FLAX_REFERENCE names the reference's sources that test also re-runs it live).
What the vectors pin: every line of the reference's own files.  What they do not: the numerics inside jax / flax
(restated by the shim in float64) and JAX's random stream (parameters and images come from this repository's seeded
numpy generators; dropout masks from oracle/philox.py, plugged in as `jax.random.bernoulli`).
"""
from __future__ import annotations

import contextlib
import importlib.util
import io
import os
import runpy
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
HERE = Path(__file__).resolve().parent
REFERENCE = Path(os.environ["VIT_FLAX_REFERENCE"]) if os.environ.get("VIT_FLAX_REFERENCE") else None
SHIM = ROOT / "oracle" / "flax_shim"

TINY = dict(image_size=32, patch_size=8, num_classes=8, dim=64, depth=2, heads=2, mlp_dim=128)
TINY_MEAN = dict(image_size=(16, 32), patch_size=(8, 16), num_classes=16, dim=64, depth=1, heads=1, mlp_dim=64)
C1 = dict(image_size=256, patch_size=32, num_classes=1000, dim=1024, depth=6, heads=16, mlp_dim=2048)
SIMPLE_TINY = dict(image_size=32, patch_size=8, num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128)
DROP_KEY = 0x1234_5678_9ABC_DEF0


def reference_available() -> bool:
    return REFERENCE is not None and (REFERENCE / "vit.py").is_file() and (REFERENCE / "simple_vit.py").is_file()


@contextlib.contextmanager
def shimmed():
    """sys.path / sys.modules with the shim's `jax` and `flax` visible, restored afterwards."""
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k.split(".")[0] in ("jax", "flax")}
    sys.path.insert(0, str(SHIM))
    try:
        yield
    finally:
        sys.path.remove(str(SHIM))
        for k in [k for k in sys.modules if k.split(".")[0] in ("jax", "flax")]:
            del sys.modules[k]
        sys.modules.update(saved)


def load_reference(stem):
    spec = importlib.util.spec_from_file_location(f"reference_{stem}", REFERENCE / f"{stem}.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def leaf_table(tree, prefix=""):
    out = []
    for k, v in tree.items():
        if isinstance(v, dict):
            out += leaf_table(v, prefix + k + "/")
        else:
            out.append((prefix + k, tuple(int(s) for s in np.shape(v))))
    return out


def philox_bernoulli():
    """`jax.random.bernoulli` that hands the reference the masks libvitb200 draws: the n-th Dropout that draws in a run is
    site n of include/vitb200.h (embedding, then per layer to_out / gelu / FF output: the reference's call order)."""
    sys.path.insert(0, str(ROOT))
    from oracle import philox

    def bernoulli(key, p, shape):
        rows = int(np.prod(shape[:-1]))
        return philox.keep_mask((rows, shape[-1]), 1.0 - float(p), key.draw_index, DROP_KEY).reshape(shape)
    return bernoulli


def run_demo(stem):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        runpy.run_path(str(REFERENCE / f"{stem}.py"), run_name="__main__")
    return buf.getvalue().strip().splitlines()


def generate():
    """-> (dict for ref_vit.npz, dict for ref_simple_vit.npz).  Needs the reference (VIT_FLAX_REFERENCE)."""
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    from _util import load_golden
    from vit_flax_b200 import init_params, perturb_params
    from vit_flax_b200.params import flatten_params
    from vit_flax_b200.simple_vit import SimpleViT as HostSimpleViT

    vit_out, simple_out = {}, {}
    with shimmed():
        import jax
        ref = load_reference("vit")
        # ---- ViT.init: the pytree the reference's own construction order produces
        v = ref.ViT(**TINY)
        tree = v.init({"params": jax.random.PRNGKey(1)}, np.zeros((1, 32, 32, 3)))["params"]
        table = leaf_table(tree)
        vit_out["init_names"] = np.array([n for n, _ in table])
        vit_out["init_shapes"] = np.array([",".join(map(str, s)) for _, s in table])
        # ---- ViT.apply on the committed inputs
        variables, meta = load_golden("tiny_cls.npz")
        vit_out["tiny_cls_logits"] = np.asarray(ref.ViT(**TINY).apply(variables, meta["images"]), dtype=np.float64)
        variables_m, meta_m = load_golden("tiny_mean.npz")
        vit_out["tiny_mean_logits"] = np.asarray(ref.ViT(pool="mean", **TINY_MEAN).apply(variables_m, meta_m["images"]),
                                                 dtype=np.float64)
        c1_vars = perturb_params(init_params(seed=1, **C1), seed=2)
        c1_img = np.random.default_rng(0).standard_normal((1, 256, 256, 3)).astype(np.float32)
        vit_out["c1_logits"] = np.asarray(ref.ViT(**C1).apply(c1_vars, c1_img), dtype=np.float64)
        # ---- dropped forward: dropout = emb_dropout = 0.1 like the README usage; masks from oracle/philox.py
        jax.random.bernoulli = philox_bernoulli()
        drop = ref.ViT(dropout=0.1, emb_dropout=0.1, **TINY)
        vit_out["tiny_cls_dropout_logits"] = np.asarray(
            drop.apply(variables, meta["images"], rngs={"dropout": jax.random.PRNGKey(DROP_KEY)}), dtype=np.float64)
        vit_out["dropout_key"] = np.uint64(DROP_KEY)
        try:
            drop.apply(variables, meta["images"])
            vit_out["dropout_without_rng_raises"] = np.bool_(False)
        except Exception as e:                     # flax: InvalidRngError
            vit_out["dropout_without_rng_raises"] = np.bool_(True)
            vit_out["dropout_without_rng_error"] = np.array(type(e).__name__)
        vit_out["demo_stdout"] = np.array(run_demo("vit"))

        # ---- simple_vit.py
        sref = load_reference("simple_vit")
        sv = sref.SimpleViT(**SIMPLE_TINY)
        img = np.random.default_rng(31).standard_normal((2, 3, 32, 32)).astype(np.float32)
        tree = sv.init({"params": jax.random.PRNGKey(1)}, img)["params"]
        table = leaf_table(tree)
        simple_out["init_names"] = np.array([n for n, _ in table])
        simple_out["init_shapes"] = np.array([",".join(map(str, s)) for _, s in table])
        host_vars = HostSimpleViT(**SIMPLE_TINY).init({"params": 5}, img)
        rng = np.random.default_rng(32)
        flat = {}
        for name, leaf in flatten_params(host_vars).items():     # make every leaf non-trivial
            leaf = np.asarray(leaf, np.float32)
            flat[name] = (leaf + 0.05 * rng.standard_normal(leaf.shape)).astype(np.float32)
        tree = {}
        for name, leaf in flat.items():
            node = tree
            parts = name.split("/")
            for p in parts[:-1]:
                node = node.setdefault(p, {})
            node[parts[-1]] = leaf
        simple_out["images"] = img
        simple_out["logits"] = np.asarray(sv.apply({"params": tree}, img), dtype=np.float64)
        for name, leaf in flat.items():
            simple_out["param." + name.replace("/", ".")] = leaf
        simple_out["demo_stdout"] = np.array(run_demo("simple_vit"))
    return vit_out, simple_out


def main():
    if not reference_available():
        raise SystemExit("set VIT_FLAX_REFERENCE to the vit_flax/ directory of a conceptofmind/vit-flax checkout: "
                         "the fixtures can only be regenerated from the reference's own files")
    vit_out, simple_out = generate()
    np.savez_compressed(HERE / "ref_vit.npz", **vit_out)
    np.savez_compressed(HERE / "ref_simple_vit.npz", **simple_out)
    print("vit.py demo:", list(vit_out["demo_stdout"]))
    print("simple_vit.py demo:", list(simple_out["demo_stdout"]))
    print("init leaves:", len(vit_out["init_names"]), "/", len(simple_out["init_names"]))


if __name__ == "__main__":
    main()
