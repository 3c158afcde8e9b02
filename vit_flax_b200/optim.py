"""``adamw``: the optimiser of the on-device training step (``ViT.trainer`` / ``SimpleViT.trainer``).

The arguments, their defaults and the arithmetic are ``optax.adamw``'s, with ``optax.clip_by_global_norm`` in front
when ``max_grad_norm`` is given and the whole chain under ``optax.apply_if_finite`` (a step whose gradients are not
all finite changes nothing).  The update itself runs in ``libvitb200.so`` (``vitb200_adamw_step``); this module only
holds and checks the hyperparameters, so it imports without a GPU.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Any, Callable, Dict, Mapping, Optional, Tuple, Union

import numpy as np

from .params import iter_leaves


def _real(name: str, v: Any) -> float:
    if isinstance(v, bool) or not isinstance(v, (int, float)) and not hasattr(v, "__float__"):
        raise ValueError(f"{name} must be a real number, got {v!r}")
    f = float(v)
    if not math.isfinite(f):
        raise ValueError(f"{name} must be finite, got {v!r}")
    return f


@dataclasses.dataclass(frozen=True)
class AdamW:
    """Checked hyperparameters of ``adamw``; build it with ``adamw(...)``."""
    learning_rate: Union[float, Callable[[int], float]]
    b1: float = 0.9
    b2: float = 0.999
    eps: float = 1e-8
    weight_decay: float = 1e-4
    mask: Any = None
    max_grad_norm: Optional[float] = None

    def lr(self, step: int) -> float:
        """The learning rate of host step ``step`` (0-based); a schedule is evaluated here, on the host."""
        v = self.learning_rate(step) if callable(self.learning_rate) else self.learning_rate
        v = _real("learning_rate", v)
        if v < 0:
            raise ValueError(f"learning_rate must be >= 0, got {v} at step {step}")
        return v

    def decay_mask(self, shapes: Mapping[str, Tuple[int, ...]]) -> Dict[str, bool]:
        """``{path: bool}`` over the leaves of a params tree (``shapes``: path -> shape, the caller's paths): where
        the weight-decay term applies.  ``mask`` None = everywhere (optax.adamw without a mask)."""
        if self.mask is None:
            return {p: True for p in shapes}
        if callable(self.mask):
            return {p: bool(self.mask(p, tuple(s))) for p, s in shapes.items()}
        return parse_mask_tree(self.mask, shapes)


def parse_mask_tree(tree: Mapping, shapes: Mapping[str, Tuple[int, ...]]) -> Dict[str, bool]:
    """A tree of bools shaped like the params tree (with or without the ``'params'`` wrapper) -> ``{path: bool}``.
    Every parameter needs an entry, and every entry must name a parameter."""
    if not isinstance(tree, Mapping):
        raise ValueError(f"mask must be None, a callable (path, shape) -> bool or a tree of bools, got {type(tree).__name__}")
    t = tree["params"] if "params" in tree and isinstance(tree["params"], Mapping) else tree
    flat = dict(iter_leaves(t))
    missing = sorted(set(shapes) - set(flat))
    extra = sorted(set(flat) - set(shapes))
    if missing or extra:
        raise ValueError(f"mask tree does not match the params tree: missing={missing[:4]} unexpected={extra[:4]}")
    out = {}
    for p, v in flat.items():
        if not isinstance(v, (bool, np.bool_)):
            raise ValueError(f"mask leaf {p!r} must be a bool, got {v!r}")
        out[p] = bool(v)
    return out


def adamw(learning_rate: Union[float, Callable[[int], float]], b1: float = 0.9, b2: float = 0.999, eps: float = 1e-8,
          weight_decay: float = 1e-4, mask: Any = None, max_grad_norm: Optional[float] = None) -> AdamW:
    """``optax.adamw`` (same names and defaults), optionally behind ``optax.clip_by_global_norm(max_grad_norm)``.

    ``learning_rate``: a float or a callable of the host step index (0 for the first ``Trainer.step``), evaluated on
    the host at every step.  Unlike optax's ``count``, the host index also advances on a step that was skipped for
    non-finite gradients (the skip is only known on the device).  ``mask``: where the weight decay applies, a callable
    ``(path, shape) -> bool`` over the flax paths of the params tree ('Transformer_0/Attention_0/Dense_0/kernel') or
    a tree of bools shaped like it.  Invalid values raise ``ValueError`` here, before any device work."""
    if not callable(learning_rate):
        lr = _real("learning_rate", learning_rate)
        if lr < 0:
            raise ValueError(f"learning_rate must be >= 0, got {learning_rate!r}")
    for name, v in (("b1", b1), ("b2", b2)):
        if not 0.0 <= _real(name, v) < 1.0:
            raise ValueError(f"{name} must be in [0, 1), got {v!r}")
    if _real("eps", eps) < 0:
        raise ValueError(f"eps must be >= 0, got {eps!r}")
    if _real("weight_decay", weight_decay) < 0:
        raise ValueError(f"weight_decay must be >= 0, got {weight_decay!r}")
    if max_grad_norm is not None and not _real("max_grad_norm", max_grad_norm) > 0:
        raise ValueError(f"max_grad_norm must be None or > 0, got {max_grad_norm!r}")
    if mask is not None and not callable(mask) and not isinstance(mask, Mapping):
        raise ValueError(f"mask must be None, a callable (path, shape) -> bool or a tree of bools, got {type(mask).__name__}")
    return AdamW(learning_rate if callable(learning_rate) else float(learning_rate), float(b1), float(b2), float(eps),
                 float(weight_decay), mask, None if max_grad_norm is None else float(max_grad_norm))
