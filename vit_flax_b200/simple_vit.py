"""``SimpleViT`` (vit_flax/simple_vit.py:99-134) on the same kernels (SURVEY.md section 8f-3).

Differences from ``ViT`` that the engine takes as configuration: NCHW images
(simple_vit.py:125), no class token, a fixed 2-D sin/cos positional table instead of a learned one
(simple_vit.py:14-25, 127-128), ``LayerNorm(epsilon=1e-5, use_bias=False)`` inside Attention /
FeedForward and in the head (simple_vit.py:41, 58, 118), a bias-free ``to_out`` (simple_vit.py:61),
mean pooling (simple_vit.py:131).  ``dim_head`` is a field here (default 64); the kernels are
built for 64.

Params pytree.  Flax names a module at CONSTRUCTION, under the module whose ``@nn.compact`` method
is running (the same rule that makes ``Attention_l`` / ``PreNorm_k`` siblings under ``Transformer_0``
in vit.py, SURVEY.md section 8c).  In simple_vit.py the ``nn.LayerNorm`` and ``nn.Dense`` handed to
``nn.Sequential([...])`` (lines 117-120) are constructed in SimpleViT's scope, before the patch
``nn.Dense`` of line 126, so the tree ``init`` gives is

    LayerNorm_0/scale [dim]          head norm          (simple_vit.py:118)
    Dense_0/{kernel [dim, classes], bias}   head        (simple_vit.py:119)
    Dense_1/{kernel [p1*p2*c, dim], bias}   patch embedding (simple_vit.py:126)
    Transformer_0/{Attention_l/{LayerNorm_0/scale, Dense_0/kernel, Dense_1/kernel},
                   FeedForward_l/{LayerNorm_0/scale, Dense_0/{kernel,bias}, Dense_1/{kernel,bias}}}

(``Sequential_0`` owns no parameters: the two layers already have a parent).  ``init`` emits this
layout.  ``apply`` / ``vjp`` also accept the ADOPTION layout that round 1 of this repository wrote
(``Dense_0`` = patch embedding, ``Sequential_0/layers_0|layers_1`` = head): the two are told apart
by the presence of ``Sequential_0`` and checked against the kernel shapes.  Neither could be checked
against a real Flax ``init`` here (jax/flax are not installable in this image): the construction-scope
layout is derived from Flax's naming rule, not executed.
"""
from __future__ import annotations

import dataclasses
from typing import Any, Dict, Optional, Tuple, Union

import numpy as np

from .params import _lecun_normal as lecun_normal, geometry, leaf_to_numpy
from .runtime import _FrontEnd, clear_cache  # noqa: F401  (the one engine cache; importable here as before)
from .vit import _seed_from_key


def posemb_sincos_2d(h: int, w: int, dim: int, temperature: float = 10000.0) -> np.ndarray:
    """simple_vit.py:14-25 -> [h*w, dim] float32."""
    assert dim % 4 == 0, "feature dimension must be multiple of 4 for sincos emb"
    y, x = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    omega = np.arange(dim // 4, dtype=np.float32) / np.float32(dim // 4 - 1)
    omega = (1.0 / (np.float32(temperature) ** omega)).astype(np.float32)
    y = y.reshape(-1, 1).astype(np.float32) * omega[None, :]
    x = x.reshape(-1, 1).astype(np.float32) * omega[None, :]
    return np.concatenate((np.sin(x), np.cos(x), np.sin(y), np.cos(y)), axis=1).astype(np.float32)


@dataclasses.dataclass(frozen=True)
class SimpleViT(_FrontEnd):
    """Same fields, order and defaults as simple_vit.py:99-108."""
    image_size: Union[int, Tuple[int, int]]
    patch_size: Union[int, Tuple[int, int]]
    num_classes: int
    dim: int
    depth: int
    heads: int
    mlp_dim: int
    channels: int = 3
    dim_head: int = 64

    def _geometry(self):
        ih, iw, ph, pw, n = geometry(self.image_size, self.patch_size)     # simple_vit.py:113-116
        if self.dim_head != 64:
            raise NotImplementedError("the attention kernels are built for dim_head = 64")
        return ih, iw, ph, pw, n

    def _validate(self, shape) -> int:
        ih, iw, _, _, _ = self._geometry()
        if len(shape) != 4 or tuple(int(s) for s in shape[1:]) != (self.channels, ih, iw):
            raise ValueError(f"expected images [B, {self.channels}, {ih}, {iw}] (NCHW, simple_vit.py:125), "
                             f"got {tuple(shape)}")
        return self.channels

    # the hooks of runtime._FrontEnd (the params tree and its two layouts are below)
    def _engine_kwargs(self, channels: int) -> Dict[str, Any]:
        ih, iw, ph, pw, _ = self._geometry()
        return dict(image_size=(ih, iw), patch_size=(ph, pw), num_classes=self.num_classes, dim=self.dim,
                    depth=self.depth, heads=self.heads, mlp_dim=self.mlp_dim, pool="mean", channels=channels,
                    nchw=True, cls_token=False, ln_eps=1e-5)

    def _param_channels(self, variables) -> int:
        return self.channels

    def _dropout_key(self, rngs) -> None:
        return None                                   # simple_vit.py has no dropout

    def _layout(self, variables) -> str:
        return self._split_tree(variables)[0]

    # ------------------------------------------------------------------ params
    def init(self, rngs: Any, x: Any) -> Dict[str, Dict]:
        """``{'params': tree}`` with the names Flax gives simple_vit.py (module docstring): LayerNorm_0 and
        Dense_0 are the head, Dense_1 the patch embedding, Transformer_0/{Attention_l, FeedForward_l}.
        Values are not bit-equal to a Flax ``init`` (that needs JAX's threefry stream); the distributions
        (lecun_normal / zeros / ones) are the reference's."""
        self._validate(np.shape(x))
        _, _, ph, pw, _ = self._geometry()
        key = rngs.get("params") if hasattr(rngs, "get") else rngs
        rng = np.random.default_rng(_seed_from_key(key))
        inner = self.dim_head * self.heads
        k0 = ph * pw * self.channels

        def dense(i, o, bias=True):
            d = {"kernel": lecun_normal(rng, (i, o))}
            if bias:
                d["bias"] = np.zeros((o,), np.float32)
            return d

        patch = dense(k0, self.dim)
        t = {}
        for l in range(self.depth):
            t[f"Attention_{l}"] = {"LayerNorm_0": {"scale": np.ones((self.dim,), np.float32)},
                                   "Dense_0": dense(self.dim, 3 * inner, False),
                                   "Dense_1": dense(inner, self.dim, False)}
            t[f"FeedForward_{l}"] = {"LayerNorm_0": {"scale": np.ones((self.dim,), np.float32)},
                                     "Dense_0": dense(self.dim, self.mlp_dim), "Dense_1": dense(self.mlp_dim, self.dim)}
        return {"params": {"LayerNorm_0": {"scale": np.ones((self.dim,), np.float32)},
                           "Dense_0": dense(self.dim, self.num_classes),
                           "Dense_1": patch, "Transformer_0": t}}

    def _split_tree(self, variables):
        """``(layout, patch_dense, transformer, head_norm, head_dense)`` of either accepted layout
        (module docstring); kernel shapes are checked so a tree of the other layout fails loudly."""
        _, _, ph, pw, _ = self._geometry()
        p = variables["params"] if "params" in variables else variables
        k0 = ph * pw * self.channels
        if "Sequential_0" in p:
            layout = "adoption"
            patch, norm, head = p["Dense_0"], p["Sequential_0"]["layers_0"], p["Sequential_0"]["layers_1"]
        else:
            layout = "construction"
            missing = [k for k in ("LayerNorm_0", "Dense_0", "Dense_1", "Transformer_0") if k not in p]
            if missing:
                raise ValueError(f"SimpleViT params tree lacks {missing}; expected LayerNorm_0 / Dense_0 (head) / "
                                 "Dense_1 (patch) / Transformer_0, or the Sequential_0 layout")
            patch, norm, head = p["Dense_1"], p["LayerNorm_0"], p["Dense_0"]
        want = {"patch": (k0, self.dim), "head": (self.dim, self.num_classes)}
        got = {"patch": tuple(np.shape(patch["kernel"])), "head": tuple(np.shape(head["kernel"]))}
        if got != want:
            raise ValueError(f"SimpleViT params ({layout} layout): kernel shapes {got} do not match the config {want}")
        return layout, patch, p["Transformer_0"], norm, head

    def _engine_tree(self, variables) -> Dict[str, Any]:
        """Re-express the SimpleViT pytree in the leaf names the engine registers (those of vit.py):
        absent biases become zeros, the sin/cos table takes the place of pos_embedding."""
        ih, iw, ph, pw, n = self._geometry()
        _, patch, tp, norm, head = self._split_tree(variables)
        z = lambda k: np.zeros((k,), np.float32)
        f = leaf_to_numpy
        t = {}
        for l in range(self.depth):
            a, ff = tp[f"Attention_{l}"], tp[f"FeedForward_{l}"]
            t[f"PreNorm_{2 * l}"] = {"LayerNorm_0": {"scale": f(a["LayerNorm_0"]["scale"]), "bias": z(self.dim)}}
            t[f"Attention_{l}"] = {"Dense_0": {"kernel": f(a["Dense_0"]["kernel"])},
                                   "Dense_1": {"kernel": f(a["Dense_1"]["kernel"]), "bias": z(self.dim)}}
            t[f"PreNorm_{2 * l + 1}"] = {"LayerNorm_0": {"scale": f(ff["LayerNorm_0"]["scale"]), "bias": z(self.dim)}}
            t[f"FeedForward_{l}"] = {"Dense_0": {k: f(v) for k, v in ff["Dense_0"].items()},
                                     "Dense_1": {k: f(v) for k, v in ff["Dense_1"].items()}}
        return {"params": {
            "pos_embedding": posemb_sincos_2d(ih // ph, iw // pw, self.dim)[None],
            "cls": np.zeros((1, 1, self.dim), np.float32),
            "Dense_0": {k: f(v) for k, v in patch.items()},
            "Transformer_0": t,
            "LayerNorm_0": {"scale": f(norm["scale"]), "bias": z(self.dim)},
            "Dense_1": {k: f(v) for k, v in head.items()}}}

    def _grads_tree(self, flat: Dict[str, np.ndarray], layout: str = "construction") -> Dict[str, Any]:
        """Engine-path leaves (vit.py leaf names: gradients, or a Trainer's weights and moments) -> the SimpleViT
        pytree in the layout the caller's params came in; the leaves SimpleViT does not have (zero biases, the fixed
        sin/cos table, the unused cls) are dropped."""
        t = {}
        for l in range(self.depth):
            pre = "Transformer_0/"
            t[f"Attention_{l}"] = {"LayerNorm_0": {"scale": flat[pre + f"PreNorm_{2 * l}/LayerNorm_0/scale"]},
                                   "Dense_0": {"kernel": flat[pre + f"Attention_{l}/Dense_0/kernel"]},
                                   "Dense_1": {"kernel": flat[pre + f"Attention_{l}/Dense_1/kernel"]}}
            t[f"FeedForward_{l}"] = {"LayerNorm_0": {"scale": flat[pre + f"PreNorm_{2 * l + 1}/LayerNorm_0/scale"]},
                                     "Dense_0": {k: flat[pre + f"FeedForward_{l}/Dense_0/{k}"] for k in ("kernel", "bias")},
                                     "Dense_1": {k: flat[pre + f"FeedForward_{l}/Dense_1/{k}"] for k in ("kernel", "bias")}}
        patch = {k: flat[f"Dense_0/{k}"] for k in ("kernel", "bias")}
        norm = {"scale": flat["LayerNorm_0/scale"]}
        head = {k: flat[f"Dense_1/{k}"] for k in ("kernel", "bias")}
        if layout == "adoption":
            return {"params": {"Dense_0": patch, "Transformer_0": t, "Sequential_0": {"layers_0": norm, "layers_1": head}}}
        return {"params": {"LayerNorm_0": norm, "Dense_0": head, "Dense_1": patch, "Transformer_0": t}}

    def vjp(self, variables: Any, img: Any, *, wrt: str = "params", precision: Optional[str] = None,
            device: Optional[int] = None, max_batch: Optional[int] = None):
        """``jax.vjp(lambda p: v.apply(p, img), variables)`` (ours; simple_vit.py never differentiates):
        ``(logits, vjp_fn)``, ``vjp_fn(dlogits)`` -> ``{'params': tree}`` of float32 gradients in SimpleViT's names.
        ``wrt="input"`` gives the float32 image gradient in the NCHW layout of ``img`` instead, ``wrt="both"``
        ``({'params': tree}, dimg)`` (``ViT.vjp``)."""
        return self._vjp(variables, img, None, wrt, precision, device, max_batch)

    def trainer(self, variables: Any, tx, *, precision: Optional[str] = None, device: Optional[int] = None,
                max_batch: Optional[int] = None):
        """``ViT.trainer`` for SimpleViT.  The fixed sin/cos table and the zero biases SimpleViT does not have are
        frozen; ``params()`` comes back in the layout ``variables`` came in."""
        from .train import Trainer
        return Trainer(self, variables, tx, precision=precision, device=device, max_batch=max_batch)

    def attention_maps(self, variables: Any, img: Any, rngs: Any = None, *, layers=None, precision: Optional[str] = None,
                       device: Optional[int] = None, max_batch: Optional[int] = None):
        """``ViT.attention_maps`` for SimpleViT: ``(logits, maps)``, ``maps`` float32 ``[B, len(layers), heads, T, T]``
        with ``T = num_patches`` (no class token); ``img`` is NCHW."""
        return self._attention_maps(variables, img, rngs, layers, precision, device, max_batch, False)

    # ------------------------------------------------------------------- apply
    def apply(self, variables: Any, img: Any, rngs: Any = None, *, precision: Optional[str] = None,
              device: Optional[int] = None, max_batch: Optional[int] = None, reload: bool = False):
        """``v.apply(params, img)`` -> logits ``[B, num_classes]`` float32; ``img`` is NCHW.  ``reload=True``
        forces the weights to be re-packed (after an in-place edit the content probe did not see)."""
        return self._apply(variables, img, rngs, precision, device, max_batch, reload)
