"""Host-side owner of one ``vitb200_model`` handle (one per device / precision).

PyTorch is plumbing here: it provides the device buffers handed to the C ABI
(``tensor.data_ptr()``) and the stream (``torch.cuda.current_stream()``).  All
compute happens inside ``libvitb200.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import numpy as np

from . import _lib
from .params import flatten_params, geometry, leaf_to_numpy


# Engine.backward(wrt=...) -> the VITB200_GRAD_* flags of vitb200_backward_ex
_WRT = {"params": _lib.GRAD_PARAMS, "input": _lib.GRAD_IMAGES, "both": _lib.GRAD_PARAMS | _lib.GRAD_IMAGES}


def _stream_ptr(torch, device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    """Create -> load_params -> forward.  Not thread-safe (like the C handle)."""

    def __init__(self, *, image_size, patch_size, num_classes, dim, depth, heads, mlp_dim,
                 pool="cls", channels=3, precision="fp16", max_batch=256, device=0,
                 dropout=0.0, emb_dropout=0.0, nchw=False, cls_token=True, ln_eps=0.0):
        import torch  # deferred: plumbing only

        if not torch.cuda.is_available():
            raise RuntimeError("vit_flax_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self._torch = torch
        self.lib = _lib.load()
        ih, iw, ph, pw, n = geometry(image_size, patch_size)
        assert pool in {"cls", "mean"}, "pool type must be either cls (cls token) or mean (mean pooling)"
        if precision not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}, got {precision!r}")
        if precision == "fp8" and (dropout or emb_dropout):
            raise ValueError("precision='fp8' is an inference forward: it is built for dropout rates 0 only")
        self.cfg = _lib.Config(
            image_h=ih, image_w=iw, patch_h=ph, patch_w=pw, channels=channels,
            num_classes=num_classes, dim=dim, depth=depth, heads=heads, mlp_dim=mlp_dim,
            pool=_lib.POOL_MEAN if pool == "mean" else _lib.POOL_CLS,
            precision=_lib.PRECISIONS[precision],
            max_batch=max_batch, dropout=float(dropout), emb_dropout=float(emb_dropout),
            flags=(_lib.FLAG_NCHW if nchw else 0) | (0 if cls_token else _lib.FLAG_NO_CLS), ln_eps=float(ln_eps))
        self.precision = precision
        self.max_batch = max_batch
        self.device = torch.device("cuda", device)
        self.tokens = n + (1 if cls_token else 0)
        self.nchw = bool(nchw)
        self.num_classes = num_classes
        self.dim = dim
        self.image_shape = (channels, ih, iw) if nchw else (ih, iw, channels)
        handle = C.c_void_p()
        _lib.check(self.lib.vitb200_create(C.byref(self.cfg), device, C.byref(handle)))
        self.handle = handle
        self._loaded = False
        # Bumped by everything that overwrites what a pending backward reads (any forward, a weight
        # reload, close): ``ViT.vjp`` captures it after ``train_forward`` and ``backward`` refuses a
        # cotangent whose forward is no longer the one held by the handle.
        self.epoch = 0

    # -- params ----------------------------------------------------------------
    def param_table(self) -> Dict[str, tuple]:
        out = {}
        n = _lib.check(self.lib.vitb200_num_params(self.handle))
        for i in range(n):
            path = C.c_char_p()
            shape = (C.c_int64 * 4)()
            nd = _lib.check(self.lib.vitb200_param_info(self.handle, i, C.byref(path), shape))
            out[path.value.decode()] = tuple(shape[:nd])
        return out

    def load_params(self, variables) -> None:
        """Upload a Flax-style params pytree (dict / FrozenDict / Mapping)."""
        self.epoch += 1
        flat = flatten_params(variables)
        table = self.param_table()
        missing = sorted(set(table) - set(flat))
        extra = sorted(set(flat) - set(table))
        if missing or extra:
            raise ValueError(f"params tree does not match the ViT config: missing={missing[:4]} "
                             f"unexpected={extra[:4]}")
        for path, leaf in flat.items():
            a = leaf_to_numpy(leaf)
            shape = (C.c_int64 * max(1, a.ndim))(*a.shape)
            _lib.check(self.lib.vitb200_set_param(self.handle, path.encode(), a.ctypes.data, shape, a.ndim))
        _lib.check(self.lib.vitb200_finalize_params(self.handle, _stream_ptr(self._torch, self.device)))
        self._loaded = True

    def set_dropout_key(self, key: int) -> None:
        """Key of the 'dropout' rng stream; the masks are a pure function of it (like Flax)."""
        _lib.check(self.lib.vitb200_set_dropout_key(self.handle, C.c_uint64(int(key) & 0xFFFFFFFFFFFFFFFF)))

    # -- forward ---------------------------------------------------------------
    def _check_images(self, shape):
        if len(shape) != 4 or tuple(shape[1:]) != self.image_shape:
            raise ValueError(f"expected images [B, {self.image_shape[0]}, {self.image_shape[1]}, "
                             f"{self.image_shape[2]}] ({'NCHW' if self.nchw else 'NHWC, channels-last'}), "
                             f"got {tuple(shape)}")
        if not 1 <= shape[0] <= self.max_batch:
            raise ValueError(f"batch {shape[0]} outside [1, max_batch={self.max_batch}]")

    def forward(self, images, out=None):
        """Device path: ``images`` fp32 CUDA tensor [B,H,W,C]; returns fp32 CUDA logits."""
        torch = self._torch
        self._check_images(images.shape)
        if images.dtype != torch.float32 or not images.is_cuda or not images.is_contiguous():
            raise ValueError("forward expects a contiguous float32 CUDA tensor")
        b = images.shape[0]
        if out is None:
            out = torch.empty((b, self.num_classes), dtype=torch.float32, device=images.device)
        self.epoch += 1
        _lib.check(self.lib.vitb200_forward(self.handle, _stream_ptr(torch, images.device),
                                            images.data_ptr(), b, out.data_ptr()))
        return out

    def forward_attn(self, images, layers, out=None, maps=None):
        """``forward`` that also records the attention weights ``softmax(q k^T * 64^-0.5)`` of ``layers`` (distinct
        indices in ``[0, depth)``, in the order given): returns ``(logits, maps)``, ``maps`` a float32 CUDA tensor
        ``[B, len(layers), heads, T, T]`` (allocated when None).  The logits are ``forward``'s."""
        torch = self._torch
        if self.precision == "fp32":
            raise ValueError("forward_attn: the fp32 validation path does not record attention maps; use 'fp16', "
                             "'bf16' or 'fp8'")
        layers = check_layers(layers, self.cfg.depth)
        self._check_images(images.shape)
        if images.dtype != torch.float32 or not images.is_cuda or not images.is_contiguous():
            raise ValueError("forward_attn expects a contiguous float32 CUDA tensor")
        b = images.shape[0]
        shape = (b, len(layers), self.cfg.heads, self.tokens, self.tokens)
        if maps is not None:
            check_maps(torch, maps, shape, images.device)
        else:
            maps = torch.empty(shape, dtype=torch.float32, device=images.device)
        if out is None:
            out = torch.empty((b, self.num_classes), dtype=torch.float32, device=images.device)
        arr = (C.c_int * len(layers))(*layers)
        self.epoch += 1
        _lib.check(self.lib.vitb200_forward_attn(self.handle, _stream_ptr(torch, images.device), images.data_ptr(), b,
                                                 out.data_ptr(), arr, len(layers), maps.data_ptr()))
        return out, maps

    # -- training (SURVEY.md section 8f-4) --------------------------------------
    def _inference_only(self, what: str) -> None:
        if self.precision == "fp8":
            raise ValueError(f"{what}: precision='fp8' is inference only; train in 'fp16' or 'bf16'")

    def train_forward(self, images, out=None):
        """Forward that keeps every activation the backward pass needs; same arguments as ``forward``.
        (The FeedForward pre-activation is rounded to 16 bits before the GELU here, so the logits can
        differ from ``forward``'s in the last 16-bit digit.)"""
        torch = self._torch
        self._inference_only("train_forward")
        self._check_images(images.shape)
        if images.dtype != torch.float32 or not images.is_cuda or not images.is_contiguous():
            raise ValueError("train_forward expects a contiguous float32 CUDA tensor")
        b = images.shape[0]
        if out is None:
            out = torch.empty((b, self.num_classes), dtype=torch.float32, device=images.device)
        self.epoch += 1
        _lib.check(self.lib.vitb200_train_forward(self.handle, _stream_ptr(torch, images.device),
                                                  images.data_ptr(), b, out.data_ptr()))
        return out

    def backward(self, dlogits, epoch: Optional[int] = None, *, wrt: str = "params", dimages=None):
        """Cotangent of the logits of the last ``train_forward`` (fp32 CUDA tensor [B, classes]) ->
        one fp32 gradient per parameter leaf, read with ``grads()`` / ``grad_tensor(path)``.
        ``epoch``: the value of ``self.epoch`` right after the ``train_forward`` this cotangent belongs
        to; a mismatch means another forward / reload ran on this engine since and is an error.
        ``wrt``: ``"params"`` (the leaf gradients), ``"input"`` (the gradient of the images only: the weight-gradient
        GEMMs are skipped, and ``grads()`` & co. raise until a backward with parameters runs) or ``"both"``.  With
        the images in ``wrt`` the image gradient is written to ``dimages`` (a contiguous float32 CUDA tensor of the
        images' shape and layout; allocated when None) and returned; otherwise None is returned."""
        torch = self._torch
        self._inference_only("backward")
        flags = _WRT.get(wrt)
        if flags is None:
            raise ValueError(f"wrt must be one of {sorted(_WRT)}, got {wrt!r}")
        if self.handle is None:
            raise RuntimeError("backward: this engine was closed (a larger batch re-created it); run vjp again")
        if epoch is not None and epoch != self.epoch:
            raise RuntimeError("backward: the engine ran another forward or reloaded its weights since the "
                               "train_forward this cotangent belongs to (activations overwritten); run vjp again")
        if dlogits.dtype != torch.float32 or not dlogits.is_cuda or not dlogits.is_contiguous() or dlogits.dim() != 2 \
                or dlogits.shape[1] != self.num_classes:
            raise ValueError(f"backward expects a contiguous float32 CUDA tensor [B, {self.num_classes}]")
        b = int(dlogits.shape[0])
        ptr = None
        if flags & _lib.GRAD_IMAGES:
            if dimages is None:
                dimages = torch.empty((b, *self.image_shape), dtype=torch.float32, device=dlogits.device)
            if dimages.dtype != torch.float32 or not dimages.is_cuda or not dimages.is_contiguous() \
                    or tuple(dimages.shape) != (b, *self.image_shape):
                raise ValueError(f"dimages must be a contiguous float32 CUDA tensor of shape {(b, *self.image_shape)}")
            ptr = dimages.data_ptr()
        _lib.check(self.lib.vitb200_backward_ex(self.handle, _stream_ptr(torch, dlogits.device),
                                                dlogits.data_ptr(), b, flags, ptr))
        return dimages if flags & _lib.GRAD_IMAGES else None

    def grad_tensor(self, path: str):
        """The gradient of one leaf as a CUDA tensor viewing the library's buffer (overwritten by the
        next ``backward``; clone it to keep it)."""
        torch = self._torch
        shape = self.param_table()[path]
        ptr = C.c_void_p()
        _lib.check(self.lib.vitb200_grad_device(self.handle, path.encode(), C.byref(ptr)))
        n = int(np.prod(shape))

        class _Buf:   # __cuda_array_interface__ view: no copy, no ownership
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(ptr.value), False), "version": 2}
        torch.cuda.current_stream(self.device).synchronize()
        return torch.as_tensor(_Buf(), device=self.device).view(*shape)

    def grads_flat(self):
        """Every leaf gradient as one contiguous fp32 CUDA tensor (a view of the library's buffer):
        what a data-parallel step all-reduces (``vit_flax_b200.dist.all_reduce_grads``)."""
        torch = self._torch
        ptr, n = C.c_void_p(), C.c_int64()
        _lib.check(self.lib.vitb200_grads_buffer(self.handle, C.byref(ptr), C.byref(n)))

        class _Buf:
            __cuda_array_interface__ = {"shape": (int(n.value),), "typestr": "<f4", "data": (int(ptr.value), False), "version": 2}
        return torch.as_tensor(_Buf(), device=self.device)

    def grads(self) -> Dict[str, np.ndarray]:
        """{flax path: float32 ndarray} of the last backward pass."""
        out = {}
        for path, shape in self.param_table().items():
            a = np.empty(shape, np.float32)
            _lib.check(self.lib.vitb200_get_grad(self.handle, _stream_ptr(self._torch, self.device),
                                                 path.encode(), a.ctypes.data))
            out[path] = a
        return out

    # -- on-device training step (vit_flax_b200.train.Trainer) --------------------
    def set_leaf_flags(self, flags: Dict[str, int]) -> None:
        """``{path: LEAF_TRAINABLE | LEAF_DECAY bits}`` for every leaf of ``param_table()``."""
        paths = list(self.param_table())
        if set(flags) != set(paths):
            raise ValueError(f"set_leaf_flags needs one entry per leaf: missing={sorted(set(paths) - set(flags))[:4]} "
                             f"unexpected={sorted(set(flags) - set(paths))[:4]}")
        arr = (C.c_uint8 * len(paths))(*[int(flags[p]) for p in paths])
        _lib.check(self.lib.vitb200_set_leaf_flags(self.handle, arr))

    def adamw_step(self, *, lr: float, b1: float, b2: float, eps: float, weight_decay: float,
                   max_grad_norm: float = 0.0, grad_scale: float = 1.0) -> None:
        """One AdamW update of the fp32 leaves from the gradient buffer of the last ``backward`` (scaled by
        ``grad_scale``), with the 16-bit weight copies re-derived in place.  Asynchronous; a pending ``vjp_fn``
        of this engine is invalidated (its forward ran on the old weights)."""
        self._inference_only("adamw_step")
        h = _lib.AdamW(lr=lr, b1=b1, b2=b2, eps=eps, weight_decay=weight_decay, max_grad_norm=max_grad_norm,
                       grad_scale=grad_scale)
        self.epoch += 1
        _lib.check(self.lib.vitb200_adamw_step(self.handle, _stream_ptr(self._torch, self.device), C.byref(h)))

    def optim_status(self):
        """``(count, skipped, grad_norm)`` of the last step; synchronises."""
        count, skipped, norm = C.c_int32(), C.c_int32(), C.c_float()
        _lib.check(self.lib.vitb200_optim_status(self.handle, _stream_ptr(self._torch, self.device),
                                                 C.byref(count), C.byref(skipped), C.byref(norm)))
        return int(count.value), int(skipped.value), float(norm.value)

    def optim_state(self):
        """``(mu, nu, count)``: CUDA tensor views of the optimiser's buffers (mu / nu flat, in the layout of
        ``grads_flat()`` and ``leaf_offsets()``; count a 1-element int32 tensor)."""
        mu, nu, cnt, n = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int64()
        _lib.check(self.lib.vitb200_optim_state(self.handle, C.byref(mu), C.byref(nu), C.byref(cnt), C.byref(n)))
        return (_device_view(self._torch, self.device, mu.value, int(n.value), "<f4"),
                _device_view(self._torch, self.device, nu.value, int(n.value), "<f4"),
                _device_view(self._torch, self.device, cnt.value, 1, "<i4"))

    def leaf_offsets(self) -> Dict[str, tuple]:
        """``{path: (element offset, shape)}`` of every leaf in the flat gradient / moment buffers (leaves in
        ``param_table`` order, each padded to a multiple of 64 elements)."""
        out, off = {}, 0
        for path, shape in self.param_table().items():
            out[path] = (off, shape)
            off += -(-int(np.prod(shape)) // 64) * 64
        return out

    def get_param(self, path: str) -> np.ndarray:
        """The current fp32 value of one leaf (after optimiser steps, the trained one); synchronises."""
        a = np.empty(self.param_table()[path], np.float32)
        _lib.check(self.lib.vitb200_get_param(self.handle, _stream_ptr(self._torch, self.device), path.encode(), a.ctypes.data))
        return a

    def softmax_xent(self, logits, labels, *, label_smoothing: float = 0.0, dscale: float = 1.0, loss=None, dlogits=None):
        """Mean softmax cross-entropy of ``logits`` (float32 CUDA [B, C]) against int32 CUDA ``labels`` [B] with
        smoothed one-hot targets, and ``dscale`` times its gradient: ``(loss 0-d tensor, dlogits [B, C])``."""
        torch = self._torch

        def ok(t, dtype, shape):
            return (isinstance(t, torch.Tensor) and t.dtype == dtype and t.is_cuda and t.is_contiguous()
                    and tuple(t.shape) == shape and t.device == logits.device)
        if not (isinstance(logits, torch.Tensor) and logits.dim() == 2):
            raise ValueError("softmax_xent expects logits as a 2-D float32 CUDA tensor [B, C]")
        b, c = int(logits.shape[0]), int(logits.shape[1])
        if not ok(logits, torch.float32, (b, c)):
            raise ValueError(f"softmax_xent expects logits as a contiguous float32 CUDA tensor [B, C], got "
                             f"{logits.dtype} {tuple(logits.shape)} on {logits.device}")
        if not ok(labels, torch.int32, (b,)):
            raise ValueError(f"softmax_xent expects labels as a contiguous int32 tensor [{b}] on {logits.device}")
        if loss is None:
            loss = torch.empty((), dtype=torch.float32, device=logits.device)
        if dlogits is None:
            dlogits = torch.empty((b, c), dtype=torch.float32, device=logits.device)
        if not ok(loss, torch.float32, ()) or not ok(dlogits, torch.float32, (b, c)):
            raise ValueError(f"softmax_xent: loss must be a 0-d and dlogits a contiguous [{b}, {c}] float32 tensor on "
                             f"{logits.device}")
        _lib.check(self.lib.vitb200_softmax_xent(_stream_ptr(torch, logits.device), logits.data_ptr(), labels.data_ptr(),
                                                 b, c, float(label_smoothing), float(dscale), loss.data_ptr(), dlogits.data_ptr()))
        return loss, dlogits

    def forward_host(self, images: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        """End-to-end path: host fp32 images in, host fp32 logits out (H2D + D2H inside)."""
        images = np.ascontiguousarray(images, dtype=np.float32)
        self._check_images(images.shape)
        b = images.shape[0]
        if out is None:
            out = np.empty((b, self.num_classes), np.float32)
        self.epoch += 1
        _lib.check(self.lib.vitb200_forward_host(self.handle, _stream_ptr(self._torch, self.device),
                                                 images.ctypes.data, b, out.ctypes.data))
        return out

    def submit_host(self, images: np.ndarray, out: np.ndarray) -> None:
        """Pipelined end-to-end path: enqueue H2D + forward + D2H of one batch and return at once
        (at most two jobs in flight; ``wait_host`` completes the oldest).  ``images`` / ``out``
        must be C-contiguous float32 (pinned for real overlap) and stay alive until waited for."""
        if images.dtype != np.float32 or not images.flags.c_contiguous:
            raise ValueError("submit_host expects a C-contiguous float32 array")
        self._check_images(images.shape)
        b = images.shape[0]
        if out.dtype != np.float32 or not out.flags.c_contiguous or out.shape != (b, self.num_classes):
            raise ValueError(f"submit_host expects a C-contiguous float32 out of shape ({b}, {self.num_classes})")
        self.epoch += 1
        _lib.check(self.lib.vitb200_submit_host(self.handle, _stream_ptr(self._torch, self.device),
                                                images.ctypes.data, b, out.ctypes.data))

    def wait_host(self) -> None:
        _lib.check(self.lib.vitb200_wait_host(self.handle))

    def forward_host_stream(self, batches):
        """Generator over host batches -> host logits, in order, two batches in flight: the H2D
        copy of batch k+1 overlaps the forward of batch k.  Logits are written into pinned
        staging arrays that are re-used two batches later: copy them if they must outlive that."""
        torch = self._torch
        outs = [torch.empty((self.max_batch, self.num_classes), dtype=torch.float32).pin_memory().numpy()
                for _ in range(2)]
        pending = []
        k = 0
        for images in batches:
            images = np.ascontiguousarray(images, dtype=np.float32)
            if len(pending) == 2:
                self.wait_host()
                yield pending.pop(0)
            out = outs[k & 1][: images.shape[0]]
            self.submit_host(images, out)
            pending.append(out)
            self._keepalive = images            # the host buffer must outlive the async copy
            k += 1
        while pending:
            self.wait_host()
            yield pending.pop(0)

    def profile_forward(self, images, out=None):
        """One forward with per-launch CUDA events -> {category: (ms, launches)}."""
        torch = self._torch
        self._check_images(images.shape)
        b = images.shape[0]
        if out is None:
            out = torch.empty((b, self.num_classes), dtype=torch.float32, device=images.device)
        n = len(_lib.CATEGORIES)
        ms = (C.c_float * n)()
        cnt = (C.c_int * n)()
        self.epoch += 1
        _lib.check(self.lib.vitb200_profile_forward(self.handle, _stream_ptr(torch, images.device),
                                                    images.data_ptr(), b, out.data_ptr(), ms, cnt))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(_lib.CATEGORIES)}

    def tokens_after_transformer(self, batch: int) -> np.ndarray:
        """The token stream ``[batch, T, dim]`` after the last block of the last forward (vit.py:157).

        Raises ``VitB200Error`` after a forward that ran the class-token tail (pool='cls', no dropout, fp16 / bf16 /
        fp8): its last block computed the class-token rows only (DESIGN.md section 3).  ``forward_attn`` with the last
        layer among ``layers`` runs that block in full, after which the stream is readable."""
        out = np.empty((batch, self.tokens, self.dim), np.float32)
        _lib.check(self.lib.vitb200_debug_tokens(self.handle, _stream_ptr(self._torch, self.device),
                                                 out.ctypes.data, batch))
        return out

    def close(self):
        if getattr(self, "handle", None):
            self.lib.vitb200_destroy(self.handle)
            self.handle = None
            self.epoch += 1

    def __del__(self):  # best effort
        try:
            self.close()
        except Exception:
            pass


def check_layers(layers, depth: int) -> List[int]:
    """The ``layers`` of an attention-map request as a list of ints: distinct, each in ``[0, depth)``, at least one;
    ``None`` means every layer.  Anything else is a ``ValueError`` (raised before any device work)."""
    if layers is None:
        return list(range(depth))
    if isinstance(layers, (int, np.integer)) or isinstance(layers, (str, bytes)):
        raise ValueError(f"layers must be a sequence of layer indices, got {layers!r}")
    out = []
    for l in layers:
        if isinstance(l, (bool, np.bool_)) or not isinstance(l, (int, np.integer)):
            raise ValueError(f"layers must hold ints, got {l!r}")
        if not 0 <= int(l) < depth:
            raise ValueError(f"layer {int(l)} outside [0, depth={depth})")
        out.append(int(l))
    if not out:
        raise ValueError("layers must name at least one layer")
    if len(set(out)) != len(out):
        raise ValueError(f"layers must be distinct, got {out}")
    return out


def check_maps(torch, maps, shape, device) -> None:
    """A caller's ``maps`` buffer must be a contiguous float32 tensor of ``shape`` on ``device``."""
    if not (isinstance(maps, torch.Tensor) and maps.dtype == torch.float32 and maps.is_contiguous()
            and tuple(maps.shape) == tuple(shape) and maps.device == torch.device(device)):
        got = f"{maps.dtype} {tuple(maps.shape)} on {maps.device}" if isinstance(maps, torch.Tensor) else type(maps).__name__
        raise ValueError(f"maps must be a contiguous float32 tensor of shape {tuple(shape)} on {device}, got {got}")


def _device_view(torch, device, ptr: int, n: int, typestr: str):
    """A CUDA tensor viewing ``n`` elements of library-owned memory (no copy, no ownership)."""
    class _Buf:
        __cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 2}
    return torch.as_tensor(_Buf(), device=device)


def launch_count() -> int:
    return int(_lib.load().vitb200_launch_count())
