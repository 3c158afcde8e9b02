"""``Trainer``: the training step of a ``ViT`` / ``SimpleViT`` on the device, built with ``model.trainer(variables, tx)``.

One ``step(x, labels)`` is ``train_forward``, the softmax cross-entropy and its gradient in one kernel, ``backward``
to the parameters, the gradient all-reduce when ``torch.distributed`` runs with more than one process, and
``vitb200_adamw_step`` (global norm, clipping, AdamW, and the 16-bit weight copies re-derived in place).  Nothing in
it waits for the GPU: the loss comes back as a 0-d CUDA tensor, the learning rate (a schedule is evaluated on the
host) and the loss scale are known on the host, and the step count lives on the device.

Loss scaling: the cotangent of a mean cross-entropy over B images is at most 1/B per logit, too small for fp16
intermediates at large B; the kernel scales it by S = 2^round(log2 B) and the optimiser divides the gradient buffer
by S (times the data-parallel world size) as it reads it.

The Trainer owns its ``Engine``.  It is not one from the cache behind ``ViT.apply``: that cache recognises a params
tree by its leaves, and after training it would otherwise hand the trained weights to ``ViT.apply(params0, x)``.
"""
from __future__ import annotations

import math
from typing import Any, Dict, Optional

import numpy as np

from . import _lib
from .checkpoint import _unflatten
from .engine import Engine
from .optim import AdamW
from .params import flatten_params, geometry, leaf_to_numpy


def _fold_in(seed: int, step: int) -> int:
    """A 64-bit key for step ``step`` of the dropout stream ``seed`` (splitmix64 of the pair)."""
    z = (seed ^ ((step + 1) * 0x9E3779B97F4A7C15)) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)


def check_labels(labels, batch: int):
    """Integer class indices of shape [batch] (numpy, anything array-like, or a torch tensor on any device) -> a
    torch tensor of them; anything else is a ValueError.  Range is not checked here: that would need the values on
    the host (the device turns an out-of-range label into a NaN loss and a skipped step)."""
    import torch
    if isinstance(labels, torch.Tensor):
        t = labels
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError(f"labels must be integers, got {t.dtype}")
    else:
        a = np.asarray(labels)
        if a.dtype.kind not in "iu":
            raise ValueError(f"labels must be integers, got {a.dtype}")
        t = torch.as_tensor(a.astype(np.int32))
    if tuple(t.shape) != (batch,):
        raise ValueError(f"labels must have shape ({batch},) (one class index per image), got {tuple(t.shape)}")
    return t


class Trainer:
    """Training state of one model on one GPU: fp32 weights, AdamW moments and step count, all on the device."""

    def __init__(self, model, variables, tx: AdamW, *, precision: Optional[str] = None, device: Optional[int] = None,
                 max_batch: Optional[int] = None):
        import torch
        from . import vit as _vit
        from .simple_vit import SimpleViT
        if not isinstance(tx, AdamW):
            raise ValueError("tx must come from vit_flax_b200.adamw(...)")
        precision = precision or _vit._DEFAULT_PRECISION
        if precision not in ("fp16", "bf16"):
            raise ValueError(f"training runs in the fp16 or bf16 precision, got {precision!r}")
        self._torch = torch
        self.model = model
        self.tx = tx
        self._simple = isinstance(model, SimpleViT)
        device = torch.cuda.current_device() if device is None else int(device)
        max_batch = 256 if max_batch is None else int(max_batch)
        if self._simple:
            ih, iw, ph, pw, _ = model._geometry()
            self._layout = model._split_tree(variables)[0]
            eng = Engine(image_size=(ih, iw), patch_size=(ph, pw), num_classes=model.num_classes, dim=model.dim,
                         depth=model.depth, heads=model.heads, mlp_dim=model.mlp_dim, pool="mean", channels=model.channels,
                         precision=precision, max_batch=max_batch, device=device, nchw=True, cls_token=False, ln_eps=1e-5)
            table = eng.param_table()
            # caller's path -> engine path; the engine leaves SimpleViT lacks (zero biases, sin/cos table, cls) are frozen
            ident = model._grads_tree({p: p for p in table}, self._layout)
            self._to_engine = dict(flatten_params(ident))
            eng.load_params(model._engine_tree(variables))
        else:
            _, _, ph, pw, _ = geometry(model.image_size, model.patch_size)
            k0 = int(np.shape(flatten_params(variables)["Dense_0/kernel"])[0])
            eng = Engine(image_size=model.image_size, patch_size=model.patch_size, num_classes=model.num_classes,
                         dim=model.dim, depth=model.depth, heads=model.heads, mlp_dim=model.mlp_dim, pool=model.pool,
                         channels=k0 // (ph * pw), precision=precision, max_batch=max_batch, device=device,
                         dropout=model.dropout, emb_dropout=model.emb_dropout)
            table = eng.param_table()
            self._to_engine = {p: p for p in table}
            eng.load_params(variables)
        self._eng = eng
        self._offsets = eng.leaf_offsets()
        decay = tx.decay_mask({cp: table[ep] for cp, ep in self._to_engine.items()})
        flags = {ep: 0 for ep in table}
        for cp, ep in self._to_engine.items():
            flags[ep] = _lib.LEAF_TRAINABLE | (_lib.LEAF_DECAY if decay[cp] else 0)
        eng.set_leaf_flags(flags)
        self._step = 0
        self._logits = torch.empty((max_batch, model.num_classes), dtype=torch.float32, device=eng.device)
        self._dlogits = torch.empty_like(self._logits)

    # ------------------------------------------------------------------ inputs
    def _images(self, x):
        torch = self._torch
        is_cuda = hasattr(x, "is_cuda") and bool(x.is_cuda)
        shape = tuple(x.shape) if hasattr(x, "shape") else np.shape(x)
        if self._simple:
            self.model._validate(shape)
        self._eng._check_images(shape)
        if is_cuda:
            return x if (x.dtype == torch.float32 and x.is_contiguous()) else x.float().contiguous()
        return torch.as_tensor(np.asarray(x, dtype=np.float32), device=self._eng.device)

    def _dropout_key(self, rngs):
        return None if self._simple else self.model._dropout_key(rngs)

    # -------------------------------------------------------------------- step
    def step(self, x, labels, *, rngs: Any = None, label_smoothing: float = 0.0):
        """One optimiser step on the batch ``(x, labels)``; returns the batch's mean loss as a 0-d CUDA tensor without
        waiting for it.  ``x`` is laid out like ``model.apply``'s images, ``labels`` holds integer class indices [B]
        (a label outside [0, num_classes) makes the loss NaN and the step is skipped).  Pass CUDA tensors for a step
        that never blocks the host: copying host arrays in synchronises.  With dropout, ``rngs={'dropout': key}``:
        step k draws its masks from ``key`` folded with k, so every step has its own."""
        ls = float(label_smoothing)
        if not 0.0 <= ls <= 1.0:
            raise ValueError(f"label_smoothing must be in [0, 1], got {label_smoothing!r}")
        b = int((x.shape if hasattr(x, "shape") else np.shape(x))[0])
        y = check_labels(labels, b)
        key = self._dropout_key(rngs)
        lr = self.tx.lr(self._step)
        x = self._images(x)
        y = y.to(device=self._eng.device, dtype=self._torch.int32).contiguous()
        eng = self._eng
        if key is not None:
            eng.set_dropout_key(_fold_in(key, self._step))
        logits = eng.train_forward(x, out=self._logits[:b])
        scale = 2.0 ** round(math.log2(b))
        loss, dl = eng.softmax_xent(logits, y, label_smoothing=ls, dscale=scale, dlogits=self._dlogits[:b])
        eng.backward(dl, wrt="params")
        world = 1
        import torch.distributed as tdist
        if tdist.is_available() and tdist.is_initialized():
            world = tdist.get_world_size()
            if world > 1:
                from .dist import all_reduce_grads
                all_reduce_grads(eng.grads_flat())
        tx = self.tx
        eng.adamw_step(lr=lr, b1=tx.b1, b2=tx.b2, eps=tx.eps, weight_decay=tx.weight_decay,
                       max_grad_norm=tx.max_grad_norm or 0.0, grad_scale=1.0 / (scale * world))
        self._step += 1
        return loss

    def apply(self, x, rngs: Any = None):
        """The forward with the current weights, like ``model.apply``: a CUDA tensor in gives CUDA logits, a host
        array numpy logits."""
        key = self._dropout_key(rngs)
        if key is not None:
            self._eng.set_dropout_key(key)
        is_cuda = hasattr(x, "is_cuda") and bool(x.is_cuda)
        xin = self._images(x)
        return self._eng.forward(xin) if is_cuda else self._eng.forward(xin).cpu().numpy()

    def last_step(self):
        """``(count, skipped, grad_norm)``: applied updates so far, whether the last step was skipped (non-finite
        gradients), and the global gradient norm it measured.  Synchronises."""
        return self._eng.optim_status()

    # ------------------------------------------------------------------ state
    def _caller_tree(self, flat: Dict[str, np.ndarray]):
        """Engine-path leaves -> ``{'params': tree}`` in the caller's layout."""
        if self._simple:
            return self.model._grads_tree(flat, self._layout)
        return {"params": _unflatten(flat)}

    def params(self) -> Dict[str, Any]:
        """``{'params': tree}`` of the current weights, numpy float32, in the layout the params came in (what
        ``save_params`` and ``model.apply`` take).  Synchronises."""
        return self._caller_tree({ep: self._eng.get_param(ep) for ep in self._offsets})

    def _split(self, buf: np.ndarray):
        return self._caller_tree({ep: buf[off: off + int(np.prod(shape))].reshape(shape).copy()
                                  for ep, (off, shape) in self._offsets.items()})

    def state_dict(self) -> Dict[str, Any]:
        """Everything a resumed run needs: params, the AdamW moments ``mu`` / ``nu`` (trees like the params),
        ``count`` (applied updates) and ``step`` (the host step index of the schedule and of the dropout keys)."""
        mu, nu, cnt = self._eng.optim_state()
        return {"params": self.params(), "mu": self._split(mu.cpu().numpy()), "nu": self._split(nu.cpu().numpy()),
                "count": int(cnt.cpu()[0]), "step": self._step}

    def load_state_dict(self, state: Dict[str, Any]) -> None:
        """Restore a ``state_dict()`` (of a Trainer of the same model and layout)."""
        torch = self._torch
        eng = self._eng
        eng.load_params(self.model._engine_tree(state["params"]) if self._simple else state["params"])
        mu, nu, cnt = eng.optim_state()
        for dst, tree in ((mu, state["mu"]), (nu, state["nu"])):
            flat = flatten_params(tree)
            buf = np.zeros(dst.shape[0], np.float32)
            for cp, ep in self._to_engine.items():
                off, shape = self._offsets[ep]
                a = leaf_to_numpy(flat[cp])
                if a.shape != tuple(shape):
                    raise ValueError(f"state {cp!r}: shape {a.shape}, expected {tuple(shape)}")
                buf[off: off + a.size] = a.ravel()
            dst.copy_(torch.from_numpy(buf))
        cnt.fill_(int(state["count"]))
        self._step = int(state["step"])
