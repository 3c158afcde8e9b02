"""Host-side mirror of the reference's ``ViT`` module surface (vit_flax/vit.py:114-167).

Same constructor fields in the same order with the same defaults, the same
``init(rngs, x)`` / ``apply(variables, x, rngs=...)`` calls and the same params
pytree, so a tree produced by the reference's Flax ``init`` loads unchanged.
Below this surface everything runs in ``libvitb200.so`` (hand-written sm_100a
kernels); there is no CPU fallback.

``dropout`` / ``emb_dropout`` > 0: the reference hard-codes ``deterministic=False``
(vit.py:50,52,83,155), so every ``apply`` drops activations and needs
``rngs={'dropout': key}`` (all four Dropout sites draw from the 'dropout' stream;
'emb_dropout' is never consumed).  Here the masks come from a Philox generator keyed by that
key -- a pure function of the key like Flax's, but not bit-equal to JAX's threefry stream.
"Dropout disabled" means the default rates 0.0, which Flax short-circuits to the identity.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Any, Dict, Optional, Tuple, Union

import numpy as np

from .params import count_params, flatten_params, geometry, init_params

# 16-bit tensor-core operand format used when `precision` is not given: "fp16" (default; same
# tcgen05 rate as bf16, 8x smaller logit error -- DESIGN.md "Operand format"), "bf16", or "fp32".
_DEFAULT_PRECISION = os.environ.get("VITB200_PRECISION", "fp16")


def _seed_from_key(key: Any) -> int:
    """Accept an int, a ``jax.random.PRNGKey``-like uint32[2], or any array-like."""
    if key is None:
        return 0
    if isinstance(key, (int, np.integer)):
        return int(key)
    a = np.asarray(key).astype(np.uint64).ravel()
    seed = 0
    for v in a:
        seed = (seed * 0x9E3779B1 + int(v)) & 0xFFFFFFFFFFFFFFFF
    return int(seed)


@dataclasses.dataclass(frozen=True)
class ViT:
    """``ViT(image_size, patch_size, num_classes, dim, depth, heads, mlp_dim, pool='cls',
    dropout=0., emb_dropout=0.)`` -- vit.py:114-125.  ``dim_head`` is a class constant
    (un-annotated in the reference, vit.py:123), so passing it is a ``TypeError`` here too."""
    image_size: Union[int, Tuple[int, int]]
    patch_size: Union[int, Tuple[int, int]]
    num_classes: int
    dim: int
    depth: int
    heads: int
    mlp_dim: int
    pool: str = "cls"
    dim_head = 64
    dropout: float = 0.0
    emb_dropout: float = 0.0

    # ------------------------------------------------------------------ helpers
    def _cfg(self, channels: int = 3) -> Dict[str, Any]:
        return dict(image_size=self.image_size, patch_size=self.patch_size,
                    num_classes=self.num_classes, dim=self.dim, depth=self.depth,
                    heads=self.heads, mlp_dim=self.mlp_dim, channels=channels)

    def _validate(self, x_shape) -> int:
        ih, iw, ph, pw, _ = geometry(self.image_size, self.patch_size)        # vit.py:130-136
        assert self.pool in {"cls", "mean"}, \
            "pool type must be either cls (cls token) or mean (mean pooling)"  # vit.py:137
        if len(x_shape) != 4:
            raise ValueError(f"expected x of rank 4 [B, H, W, C] (channels-last), got shape {tuple(x_shape)}")
        b, h, w, c = (int(s) for s in x_shape)
        if (h, w) != (ih, iw):
            hint = " (looks like NCHW; the reference takes NHWC, vit.py:146)" if (w, c) == (ih, iw) else ""
            raise ValueError(f"expected images of {ih}x{iw}, got {h}x{w}{hint}")
        return c

    def _dropout_key(self, rngs):
        """None when both rates are 0 (Flax draws nothing); else the 'dropout' key, required like in
        Flax, where ``apply`` without it fails with "Dropout_0 needs PRNG for 'dropout'"."""
        if self.dropout == 0.0 and self.emb_dropout == 0.0:
            return None
        if not (0.0 <= self.dropout < 1.0 and 0.0 <= self.emb_dropout < 1.0):
            raise ValueError("dropout rates must be in [0, 1)")
        key = rngs.get("dropout") if hasattr(rngs, "get") else None
        if key is None:
            raise ValueError("ViT was built with dropout > 0 and the reference applies it on every call "
                             "(deterministic=False): pass rngs={'dropout': key}")
        return _seed_from_key(key)

    def num_params(self, channels: int = 3) -> int:
        """What the reference's demo prints (vit.py:195-197)."""
        return count_params(**self._cfg(channels))

    # --------------------------------------------------------------------- init
    def init(self, rngs: Any, x: Any) -> Dict[str, Dict]:
        """``v.init({'params': key, 'dropout': key, 'emb_dropout': key}, img)`` (vit.py:187-191).

        Returns ``{'params': tree}`` with the reference's names, shapes, dtypes
        (float32) and initialiser distributions (zeros for pos_embedding / cls /
        biases, ones for LayerNorm scales, lecun_normal for Dense kernels)."""
        channels = self._validate(np.shape(x))
        key = rngs.get("params") if hasattr(rngs, "get") else rngs
        return init_params(seed=_seed_from_key(key), **self._cfg(channels))

    # -------------------------------------------------------------------- apply
    def apply(self, variables: Any, x: Any, rngs: Any = None, *, precision: Optional[str] = None,
              device: Optional[int] = None, max_batch: Optional[int] = None, reload: bool = False):
        """``v.apply(params, img, rngs=init_rngs)`` -> logits ``[B, num_classes]`` float32.

        ``x``: ``[B, H, W, C]`` channels-last float32.  A host array (numpy or
        anything ``np.asarray``-able) is copied to the GPU and the logits come
        back as a numpy array; a CUDA ``torch.Tensor`` stays on the device and
        a CUDA tensor is returned.  ``rngs`` is accepted and ignored at dropout
        rate 0 (Flax draws nothing there).  Keyword-only extras are ours:
        ``precision`` ('fp16' / 'bf16' tcgen05 paths, 'fp8' -- E4M3 operands on to_qkv and the FeedForward,
        inference only, DESIGN.md -- and 'fp32', the validation path)."""
        eng, xin = self._forward_engine(variables, x, rngs, precision, device, max_batch, reload)
        if xin is not None:
            return eng.forward(xin)
        return eng.forward_host(np.asarray(x, dtype=np.float32))

    def _forward_engine(self, variables, x, rngs, precision, device, max_batch, reload):
        """What ``apply`` and ``attention_maps`` share: the dropout key (checked first), the image checks, the device,
        the cached engine with ``variables`` loaded and the key set.  Returns ``(engine, x as a contiguous float32 CUDA
        tensor)`` for a CUDA ``x``, ``(engine, None)`` for a host array."""
        from .runtime import get_engine   # deferred: needs torch + CUDA
        key = self._dropout_key(rngs)
        is_torch_cuda = hasattr(x, "is_cuda") and bool(x.is_cuda)
        channels = self._validate(tuple(x.shape) if hasattr(x, "shape") else np.shape(x))
        batch = int(x.shape[0])
        if device is None:
            device = x.device.index if is_torch_cuda and x.device.index is not None else _current_device()
        eng = get_engine(self, channels, precision or _DEFAULT_PRECISION, device, max_batch or batch, variables, reload)
        if key is not None:
            eng.set_dropout_key(key)
        if not is_torch_cuda:
            return eng, None
        import torch
        return eng, (x if (x.dtype == torch.float32 and x.is_contiguous()) else x.float().contiguous())

    def attention_maps(self, variables: Any, x: Any, rngs: Any = None, *, layers=None, precision: Optional[str] = None,
                       device: Optional[int] = None, max_batch: Optional[int] = None, reload: bool = False):
        """``apply`` that also returns the attention weights ``softmax(q k^T * dim_head^-0.5)`` (vit.py:73-75) of
        ``layers`` (ours; vit-pytorch's ``Recorder`` returns the same): ``(logits, maps)``, ``maps`` float32
        ``[B, len(layers), heads, T, T]`` with ``T = num_patches + 1`` (the class token is row and column 0).

        ``layers``: distinct layer indices in ``[0, depth)``, recorded in the order given; default every layer.
        ``logits`` are ``apply``'s, bit for bit.  A CUDA tensor in gives CUDA tensors out, a host array numpy.  With
        dropout > 0 pass ``rngs={'dropout': key}`` as for ``apply``: the maps are those of that dropped forward (the
        reference drops no attention weights, vit.py:75-83).  The maps are recomputed on the tensor cores from the
        16-bit q / k of the forward (precision 'fp16', 'bf16' or 'fp8'); 'fp32' is refused.  ``reload`` as for ``apply``."""
        from .engine import check_layers
        if (precision or _DEFAULT_PRECISION) == "fp32":
            raise ValueError("attention_maps: the fp32 validation path does not record attention maps; use 'fp16', "
                             "'bf16' or 'fp8'")
        layers = check_layers(layers, self.depth)
        eng, xin = self._forward_engine(variables, x, rngs, precision, device, max_batch, reload)
        if xin is not None:
            return eng.forward_attn(xin, layers)
        import torch
        logits, maps = eng.forward_attn(torch.as_tensor(np.asarray(x, dtype=np.float32), device=eng.device), layers)
        return logits.cpu().numpy(), maps.cpu().numpy()

    def vjp(self, variables: Any, x: Any, rngs: Any = None, *, wrt: str = "params", precision: Optional[str] = None,
            device: Optional[int] = None, max_batch: Optional[int] = None):
        """``jax.vjp(lambda p: v.apply(p, x), variables)`` (ours: nothing in the reference trains).

        Returns ``(logits, vjp_fn)``; ``vjp_fn(dlogits)`` gives ``{'params': tree}`` of float32
        gradients with the reference's names and shapes.  Host arrays in -> numpy out, CUDA tensors
        in -> CUDA logits out (gradients always come back as numpy).  With fp16 operands the
        cotangent is scaled to unit magnitude on the way in and the gradients back on the way out
        (loss scaling: the map is linear).  With dropout rates > 0 pass ``rngs={'dropout': key}``: the
        forward drops with that key's masks and ``vjp_fn`` differentiates that same dropped forward.

        ``wrt`` picks what ``vjp_fn`` differentiates with respect to: ``"params"`` (the default, above),
        ``"input"`` -- ``dx``, the float32 gradient of the images with the shape of ``x`` (saliency maps,
        FGSM / PGD); the weight-gradient GEMMs are skipped -- or ``"both"`` -- ``({'params': tree}, dx)``, the
        order of ``jax.vjp(v.apply, variables, x)``.  ``dx`` is a CUDA tensor when ``x`` is one, numpy otherwise."""
        want_params, want_input = _parse_wrt(wrt)
        _check_trainable_precision(precision or _DEFAULT_PRECISION, "vjp")
        from .runtime import get_engine
        import torch
        key = self._dropout_key(rngs)          # rates > 0 need rngs={'dropout': key}, like apply
        is_torch_cuda = hasattr(x, "is_cuda") and bool(x.is_cuda)
        channels = self._validate(tuple(x.shape) if hasattr(x, "shape") else np.shape(x))
        batch = int(x.shape[0])
        if device is None:
            device = x.device.index if is_torch_cuda and x.device.index is not None else _current_device()
        eng = get_engine(self, channels, precision or _DEFAULT_PRECISION, device, max_batch or batch, variables, False)
        dev = torch.device("cuda", device)
        xin = x if is_torch_cuda else torch.as_tensor(np.asarray(x, dtype=np.float32), device=dev)
        xin = xin if (xin.dtype == torch.float32 and xin.is_contiguous()) else xin.float().contiguous()
        if key is not None:
            eng.set_dropout_key(key)           # the backward replays the masks of this key
        logits = eng.train_forward(xin)
        epoch = eng.epoch      # any later forward / reload on this engine invalidates vjp_fn

        def vjp_fn(dlogits):
            d = dlogits if hasattr(dlogits, "is_cuda") else torch.as_tensor(np.asarray(dlogits, dtype=np.float32))
            d = d.to(device=dev, dtype=torch.float32).contiguous()
            if tuple(d.shape) != (batch, self.num_classes):
                raise ValueError(f"vjp_fn expects a cotangent of shape ({batch}, {self.num_classes})")
            peak = float(d.abs().max())
            scale = 1.0 if peak == 0.0 or not np.isfinite(peak) else float(2.0 ** -np.round(np.log2(peak)))
            dx = eng.backward(d * scale if scale != 1.0 else d, epoch=epoch, wrt=wrt)
            out = []
            if want_params:
                from .checkpoint import _unflatten
                out.append({"params": _unflatten({k: g / np.float32(scale) for k, g in eng.grads().items()})})
            if want_input:
                out.append(_unscale_images(dx, scale, is_torch_cuda))
            return out[0] if len(out) == 1 else tuple(out)

        return (logits if is_torch_cuda else logits.cpu().numpy()), vjp_fn

    def trainer(self, variables: Any, tx, *, precision: Optional[str] = None, device: Optional[int] = None,
                max_batch: Optional[int] = None):
        """A ``Trainer`` (vit_flax_b200/train.py) that fine-tunes ``variables`` with ``tx`` (``vit_flax_b200.adamw``)
        entirely on the device (ours: nothing in the reference trains).  ``max_batch``: the largest batch ``step``
        will see (default 256).  The trainer owns its weights: ``apply(variables, x)`` still runs ``variables``."""
        from .train import Trainer
        return Trainer(self, variables, tx, precision=precision, device=device, max_batch=max_batch)

    def apply_stream(self, variables: Any, batches, *, precision: Optional[str] = None,
                     device: Optional[int] = None, max_batch: int = 256):
        """Serving-style extension of ``apply`` (ours, not in the reference): iterate host batches
        ``[B, H, W, C]`` float32 and yield their logits in order, keeping two batches in flight so the
        host->device copy of the next batch overlaps the forward of the current one.  Yielded arrays
        are staging buffers re-used two batches later."""
        if self.dropout != 0.0 or self.emb_dropout != 0.0:
            raise NotImplementedError("apply_stream is an inference path: construct ViT with the default rates 0.0")
        from .runtime import get_engine

        it = iter(batches)
        try:
            first = next(it)
        except StopIteration:
            return
        channels = self._validate(np.shape(first))
        if device is None:
            device = _current_device()
        eng = get_engine(self, channels, precision or _DEFAULT_PRECISION, device, max_batch, variables, False)

        def chain():
            yield first
            for b in it:
                self._validate(np.shape(b))
                yield b
        yield from eng.forward_host_stream(chain())

    def __call__(self, *a, **k):  # flax modules are called through init/apply
        raise TypeError("call ViT through .init(rngs, x) / .apply(variables, x), like the flax module")


def _parse_wrt(wrt: str) -> Tuple[bool, bool]:
    """``vjp(wrt=...)`` -> (parameter gradients?, image gradient?); checked before any device work."""
    choices = {"params": (True, False), "input": (False, True), "both": (True, True)}
    if wrt not in choices:
        raise ValueError(f"wrt must be one of 'params', 'input' or 'both', got {wrt!r}")
    return choices[wrt]


def _check_trainable_precision(precision: str, what: str) -> None:
    """fp8 is an inference forward: refused before any device work by everything that differentiates."""
    if precision == "fp8":
        raise ValueError(f"{what}: precision='fp8' is inference only; use 'fp16' or 'bf16' to differentiate or train")


def _unscale_images(dx, scale: float, as_cuda: bool):
    """Undo the power-of-two cotangent scaling on an image gradient (exact) and hand it out like the logits."""
    if scale != 1.0:
        dx.div_(scale)
    return dx if as_cuda else dx.cpu().numpy()


def _current_device() -> int:
    import torch
    return torch.cuda.current_device()


def tree_shapes(variables) -> Dict[str, Tuple[int, ...]]:
    return {k: tuple(np.shape(v)) for k, v in flatten_params(variables).items()}
