"""The checker of image gradients: ``jax.vjp(v.apply, params, x)[1](dlogits)`` restated as float64 torch autograd
through ``oracle.vit_torch``'s forward, with the images as a differentiated leaf next to the parameters.  It is
``oracle.vit_torch.vit_vjp`` plus the image gradient; the parameter gradients are computed by the same graph."""
import torch

from oracle import vit_torch


def vit_vjp_images(variables, images, dlogits, *, dtype=torch.float64, **cfg):
    """-> ``(logits, grads, dimages)`` as numpy: ``grads`` shaped like ``variables['params']``, ``dimages`` like
    ``images`` (NHWC)."""
    tree = variables["params"] if "params" in variables else variables

    def conv(t):
        if isinstance(t, dict) or hasattr(t, "items"):
            return {k: conv(v) for k, v in t.items()}
        return torch.as_tensor(t).to(dtype).clone().requires_grad_(True)

    p = conv(tree)
    x = torch.as_tensor(images).to(dtype).clone().requires_grad_(True)
    with torch.enable_grad():
        logits = vit_torch._vit_forward({"params": p}, x, **cfg)
        (logits * torch.as_tensor(dlogits).to(dtype)).sum().backward()

    def grads(t):
        if isinstance(t, dict):
            return {k: grads(v) for k, v in t.items()}
        return (t.grad if t.grad is not None else torch.zeros_like(t)).detach().numpy()

    return logits.detach().numpy(), grads(p), x.grad.detach().numpy()
