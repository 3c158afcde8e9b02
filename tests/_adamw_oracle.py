"""float64 numpy references of the on-device training step: optax-style AdamW behind clip_by_global_norm and
apply_if_finite, and softmax cross-entropy with smoothed labels.  Checked against torch.optim.AdamW and torch
autograd in tests/test_optim.py; the GPU tests hold the kernels to them."""
import numpy as np


def adamw_ref(params, grads, mu, nu, count, *, lr, b1=0.9, b2=0.999, eps=1e-8, weight_decay=1e-4, decay=None,
              trainable=None, max_grad_norm=0.0, grad_scale=1.0):
    """One step on dicts of arrays (path -> array).  ``decay`` / ``trainable``: path -> bool (default all True).
    Returns ``(params, mu, nu, count, skipped, norm)``, new float64 dicts; frozen leaves are returned unchanged."""
    keys = [k for k in params if trainable is None or trainable[k]]
    g = {k: np.asarray(grads[k], np.float64) * grad_scale for k in keys}
    finite = all(np.isfinite(v).all() for v in g.values())
    norm = float(np.sqrt(sum(float((v * v).sum()) for v in g.values()))) if finite else float("nan")
    p2 = {k: np.asarray(v, np.float64).copy() for k, v in params.items()}
    m2 = {k: np.asarray(v, np.float64).copy() for k, v in mu.items()}
    n2 = {k: np.asarray(v, np.float64).copy() for k, v in nu.items()}
    if not finite:
        return p2, m2, n2, count, 1, norm
    clip = max_grad_norm / max(norm, max_grad_norm) if max_grad_norm > 0 else 1.0
    t = count + 1
    bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
    for k in keys:
        gk = g[k] * clip
        m2[k] = b1 * m2[k] + (1 - b1) * gk
        n2[k] = b2 * n2[k] + (1 - b2) * gk * gk
        u = (m2[k] / bc1) / (np.sqrt(n2[k] / bc2) + eps)
        if decay is None or decay[k]:
            u = u + weight_decay * p2[k]
        p2[k] = p2[k] - lr * u
    return p2, m2, n2, t, 0, norm


def xent_ref(logits, labels, label_smoothing=0.0, dscale=1.0):
    """mean_b sum_c -q log_softmax(z_b) with q = (1 - eps) onehot + eps / C, and dscale * its gradient (float64)."""
    z = np.asarray(logits, np.float64)
    b, c = z.shape
    q = np.full((b, c), label_smoothing / c)
    q[np.arange(b), np.asarray(labels)] += 1.0 - label_smoothing
    m = z.max(axis=1, keepdims=True)
    logp = z - m - np.log(np.exp(z - m).sum(axis=1, keepdims=True))
    loss = float(-(q * logp).sum() / b)
    return loss, dscale * (np.exp(logp) - q) / b
