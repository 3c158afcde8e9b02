"""What ``ViT`` and ``SimpleViT`` share above the ``Engine``: the engine cache and one implementation each of
``apply``, ``attention_maps`` and ``vjp`` (``_FrontEnd``), written against the few hooks by which the two models
differ.

The cache keeps one ``Engine`` per (model, channels, precision, device) -- the models are frozen dataclasses, so
equal configurations share an engine and a ``ViT`` never shares one with a ``SimpleViT`` -- re-creates it when a
larger batch comes, and re-packs the weights only when different params are passed.

"Different" is decided by ``ParamsStamp`` over the caller's tree: the leaves of the last loaded tree are held by
STRONG reference and compared with ``is`` (an ``id()`` alone can be recycled by CPython as soon as the old object
dies -- ``v.apply({'params': p1}, x); v.apply({'params': p2}, x)`` builds two temporaries with the same id), plus a
cheap content probe per leaf (a strided sample of up to 16 values for host arrays, the ``_version`` counter for
torch tensors), so the usual in-place updates -- an optimiser step, ``leaf *= 0`` -- are seen too.  An in-place
edit that misses every probed element of a host array is the one case left to ``reload=True``.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple

import numpy as np

from .engine import Engine, check_layers
from .params import flatten_params

# 16-bit tensor-core operand format used when `precision` is not given: "fp16" (default; same
# tcgen05 rate as bf16, 8x smaller logit error -- DESIGN.md "Operand format"), "bf16", or "fp32".
_DEFAULT_PRECISION = os.environ.get("VITB200_PRECISION", "fp16")

_engines: Dict[Tuple, Tuple[Engine, Optional["ParamsStamp"]]] = {}

_PROBE = 16   # sampled values per host leaf


def _probe(leaf) -> object:
    """Cheap content witness of one leaf (never copies the leaf, never synchronises a GPU)."""
    if hasattr(leaf, "_version") and hasattr(leaf, "data_ptr"):         # torch.Tensor (any device)
        return ("torch", int(leaf._version), int(leaf.data_ptr()))
    if isinstance(leaf, np.ndarray):
        flat = leaf.reshape(-1) if leaf.flags.c_contiguous else leaf.ravel()
        n = flat.size
        if n == 0:
            return ("np", b"")
        step = max(1, n // _PROBE)
        return ("np", flat[::step][:_PROBE].tobytes(), flat[-1:].tobytes())
    return ("other",)                                                    # jax arrays are immutable: identity is enough


class ParamsStamp:
    """Identity (strong references, compared with ``is``) + content probe of a params tree."""

    def __init__(self, variables):
        flat = flatten_params(variables)
        self.keys: List[str] = sorted(flat)
        self.leaves = [flat[k] for k in self.keys]       # strong references: ids cannot be recycled
        self.probes = [_probe(v) for v in self.leaves]

    def matches(self, other: Optional["ParamsStamp"]) -> bool:
        if other is None or self.keys != other.keys:
            return False
        return all(a is b for a, b in zip(self.leaves, other.leaves)) and self.probes == other.probes


def _new_engine(model, channels: int, precision: str, device: int, max_batch: int) -> Engine:
    """An ``Engine`` for ``model`` (no weights loaded), outside the cache."""
    return Engine(**model._engine_kwargs(channels), precision=precision, max_batch=max_batch, device=device)


def get_engine(model, channels: int, precision: str, device: int, batch: int, variables,
               reload: bool = False) -> Engine:
    """The cached engine of ``model`` holding ``variables`` (the caller's tree), for batches up to ``batch``."""
    key = (model, channels, precision, device)
    eng, loaded = _engines.get(key, (None, None))
    if eng is None or eng.max_batch < batch:
        if eng is not None:
            eng.close()
        eng, loaded = _new_engine(model, channels, precision, device, batch), None
    stamp = ParamsStamp(variables)
    if reload or not stamp.matches(loaded):
        _engines[key] = (eng, None)               # a load that fails part-way leaves no stale stamp behind
        eng.load_params(model._engine_tree(variables))
        loaded = stamp
    _engines[key] = (eng, loaded)
    return eng


def clear_cache() -> None:
    for eng, _ in _engines.values():
        eng.close()
    _engines.clear()


def _is_cuda(x) -> bool:
    return hasattr(x, "is_cuda") and bool(x.is_cuda)


def _device_images(eng: Engine, x):
    """``x`` as a contiguous float32 CUDA tensor: a host array is copied to ``eng``'s device, a CUDA tensor is
    converted only when it is not one already."""
    import torch
    if not _is_cuda(x):
        x = torch.as_tensor(np.asarray(x, dtype=np.float32), device=eng.device)
    return x if (x.dtype == torch.float32 and x.is_contiguous()) else x.float().contiguous()


class _FrontEnd:
    """``apply`` / ``attention_maps`` / ``vjp`` of ``ViT`` and ``SimpleViT``.  A model says how it differs through:

    * ``_dropout_key(rngs)``: the dropout seed, or None when the model draws no masks; checked first;
    * ``_validate(shape)``: the image checks, returning the channel count;
    * ``_engine_kwargs(channels)``: the ``Engine`` configuration (everything but precision, batch and device);
    * ``_engine_tree(variables)``: the caller's params tree in the engine's leaf names;
    * ``_layout(variables)`` / ``_grads_tree(flat, layout)``: which layout the caller's tree is in, and engine-path
      leaves back as ``{'params': tree}`` in that layout."""

    def _engine(self, variables, x, rngs, precision, device, max_batch, reload) -> Engine:
        """Argument checks, then the cached engine with ``variables`` loaded and the dropout key set."""
        key = self._dropout_key(rngs)
        channels = self._validate(np.shape(x))
        if device is None:
            import torch
            device = x.device.index if _is_cuda(x) and x.device.index is not None else torch.cuda.current_device()
        eng = get_engine(self, channels, precision, device, max_batch or int(x.shape[0]), variables, reload)
        if key is not None:
            eng.set_dropout_key(key)
        return eng

    def _apply(self, variables, x, rngs, precision, device, max_batch, reload):
        eng = self._engine(variables, x, rngs, precision or _DEFAULT_PRECISION, device, max_batch, reload)
        if _is_cuda(x):
            return eng.forward(_device_images(eng, x))
        return eng.forward_host(np.asarray(x, dtype=np.float32))

    def _attention_maps(self, variables, x, rngs, layers, precision, device, max_batch, reload):
        precision = precision or _DEFAULT_PRECISION
        if precision == "fp32":
            raise ValueError("attention_maps: the fp32 validation path does not record attention maps; use 'fp16', "
                             "'bf16' or 'fp8'")
        layers = check_layers(layers, self.depth)
        eng = self._engine(variables, x, rngs, precision, device, max_batch, reload)
        logits, maps = eng.forward_attn(_device_images(eng, x), layers)
        return (logits, maps) if _is_cuda(x) else (logits.cpu().numpy(), maps.cpu().numpy())

    def _vjp(self, variables, x, rngs, wrt, precision, device, max_batch):
        choices = {"params": (True, False), "input": (False, True), "both": (True, True)}
        if wrt not in choices:
            raise ValueError(f"wrt must be one of 'params', 'input' or 'both', got {wrt!r}")
        want_params, want_input = choices[wrt]
        precision = precision or _DEFAULT_PRECISION
        if precision == "fp8":
            raise ValueError("vjp: precision='fp8' is inference only; use 'fp16' or 'bf16' to differentiate or train")
        import torch
        eng = self._engine(variables, x, rngs, precision, device, max_batch, False)
        layout = self._layout(variables)
        batch, cuda = int(x.shape[0]), _is_cuda(x)
        logits = eng.train_forward(_device_images(eng, x))    # with dropout, the backward replays this key's masks
        epoch = eng.epoch      # any later forward / reload on this engine invalidates vjp_fn

        def vjp_fn(dlogits):
            d = dlogits if hasattr(dlogits, "is_cuda") else torch.as_tensor(np.asarray(dlogits, dtype=np.float32))
            d = d.to(device=eng.device, dtype=torch.float32).contiguous()
            if tuple(d.shape) != (batch, self.num_classes):
                raise ValueError(f"vjp_fn expects a cotangent of shape ({batch}, {self.num_classes})")
            # loss scaling: the cotangent goes in at unit magnitude (a power of two, so undoing it is exact)
            peak = float(d.abs().max())
            scale = 1.0 if peak == 0.0 or not np.isfinite(peak) else float(2.0 ** -np.round(np.log2(peak)))
            dx = eng.backward(d * scale if scale != 1.0 else d, epoch=epoch, wrt=wrt)
            out = []
            if want_params:
                out.append(self._grads_tree({k: g / np.float32(scale) for k, g in eng.grads().items()}, layout))
            if want_input:
                if scale != 1.0:
                    dx.div_(scale)
                out.append(dx if cuda else dx.cpu().numpy())
            return out[0] if len(out) == 1 else tuple(out)

        return (logits if cuda else logits.cpu().numpy()), vjp_fn
