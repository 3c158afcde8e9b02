"""The float64 references of the backward kernels (tests/_bwd_ref.py), checked on the CPU: against torch autograd with
rounding off, against oracle/philox.py for the dropout masks, and against mutants -- each plausible kernel bug must land
well outside the bound the GPU tests (tests/test_gpu_backward_kernels.py) use."""
import numpy as np
import pytest
import torch

import _bwd_ref as R
from oracle import philox


def _attn_inputs(B, T, heads, tdt, seed):
    g = torch.Generator().manual_seed(seed)
    inner = heads * 64
    qkv = (torch.randn((B, T, 3 * inner), generator=g, dtype=torch.float64) * 1.2)
    do = torch.randn((B, T, inner), generator=g, dtype=torch.float64)
    if tdt is not None:
        qkv, do = R.rnd(qkv, tdt), R.rnd(do, tdt)
    q, k, v = qkv.view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    o = (torch.softmax(q @ k.transpose(-1, -2) / 8, -1) @ v).permute(0, 2, 1, 3).reshape(B, T, inner)
    return qkv, R.rnd(o, tdt), do


def _autograd_attention(qkv, do, heads):
    B, T, _ = qkv.shape
    x = qkv.view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4).contiguous().requires_grad_(True)
    o = torch.softmax(x[0] @ x[1].transpose(-1, -2) / 8.0, dim=-1) @ x[2]
    (o * do.view(B, T, heads, 64).permute(0, 2, 1, 3)).sum().backward()
    return x.grad.permute(1, 3, 0, 2, 4).reshape(B, T, -1)


def test_keep_mask_is_the_philox_of_the_oracle():
    for rows, cols, rate, site, key in [(3, 8, 0.5, 0, 0x1234), (37, 264, 0.1, 7, 0xFEEDFACE12345678), (1, 5, 0.3, 2, 1 << 40)]:
        got = R.keep_mask(rows, cols, rate, site, key, "cpu").numpy()
        np.testing.assert_array_equal(got, philox.keep_mask((rows, cols), rate, site, key))
    assert R.inv_keep(0.5) == 2.0


@pytest.mark.parametrize("B,T,heads", [(2, 17, 2), (1, 197, 1), (1, 300, 2)])
def test_attention_ref_without_rounding_is_autograd(B, T, heads):
    qkv, o, do = _attn_inputs(B, T, heads, None, T)
    got, _ = R.attention_bwd(qkv, o, do, heads, None)
    want = _autograd_attention(qkv, do, heads)
    assert (got - want).abs().max().item() < 1e-12 * max(1.0, want.abs().max().item())


@pytest.mark.parametrize("B,T,heads", [(2, 197, 2), (1, 257, 2), (1, 1025, 1)])
@pytest.mark.parametrize("fmt,floor_max", [("fp16", 1.5e-2), ("bf16", 5e-2)])
def test_attention_ref_floor_of_the_format(B, T, heads, fmt, floor_max):
    """The same-rounding reference against the exact adjoint: the 16-bit roundings of P, dS and the outputs alone move
    dqkv by this much (max error / max |exact|); it stays inside the end-to-end bound of test_attention_bwd.  Measured:
    fp16 5e-4 to 6e-4, bf16 3e-3 to 4e-3 at these shapes."""
    tdt = {"fp16": torch.float16, "bf16": torch.bfloat16}[fmt]
    qkv, o, do = _attn_inputs(B, T, heads, tdt, T + 1)
    got, _ = R.attention_bwd(qkv, o, do, heads, tdt)
    want = _autograd_attention(qkv, do, heads)
    floor = ((got - want).abs().max() / want.abs().max()).item()
    assert 0 < floor < floor_max / 3, floor


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_attention_bound_catches_mutants(fmt):
    """Streamed shape (T = 300: key tiles 0..2).  Each mutant of the reference must exceed the bound by a clear margin
    (max |mutant - ref| / bound > 4).  D from the exact O instead of O16 differs by about u |dO| |O| per row, which the
    bound covers: that slip is below what a comparison with any fp32 kernel can resolve, so it is asserted to stay
    inside the bound rather than outside."""
    tdt = {"fp16": torch.float16, "bf16": torch.bfloat16}[fmt]
    qkv, o, do = _attn_inputs(2, 300, 2, tdt, 5)
    ref, bound = R.attention_bwd(qkv, o, do, 2, tdt)
    ratio = lambda m: ((R.attention_bwd(qkv, o, do, 2, tdt, mutant=m)[0] - ref).abs() / bound).max().item()
    assert ratio("dq_key_tile") > 4
    assert ratio("lse_shift") > 4
    assert ratio("d_exact_o") <= 1.0


def test_ln_ref_is_autograd_and_its_bound_catches_a_skipped_row():
    g = torch.Generator().manual_seed(3)
    rows, dim = 37, 260
    x = torch.randn((rows, dim), generator=g, dtype=torch.float64) * 2 + 0.5
    gamma = torch.randn(dim, generator=g, dtype=torch.float64) * 0.5 + 1
    dy = R.dyadic((rows, dim), 4, g, "cpu").double()
    dx, dgamma, dbeta, bdx, bdg = R.ln_bwd(x, gamma, dy)
    xr, gr = x.clone().requires_grad_(True), gamma.clone().requires_grad_(True)
    br = torch.zeros(dim, dtype=torch.float64, requires_grad=True)
    (torch.nn.functional.layer_norm(xr, (dim,), gr, br, eps=1e-6) * dy).sum().backward()
    assert (dx - xr.grad).abs().max() < 1e-12 and (dgamma - gr.grad).abs().max() < 1e-11 and (dbeta - br.grad).abs().max() < 1e-12
    skipped = dx.clone()
    skipped[-1] = 0                                                  # the last (ragged) row never written
    assert ((skipped - dx).abs() / bdx).max() > 1e3
    xhat = R.ln_stats(x)[2]
    assert (((dy[:-1] * xhat[:-1]).sum(0) - dgamma).abs() / bdg).max() > 4
    assert not torch.equal(dy[:-1].sum(0), dbeta)                  # dbeta is checked bit for bit


def test_colsum_exactness_catches_a_missing_row_and_a_missing_mask():
    g = torch.Generator().manual_seed(4)
    rows, cols, rate, site, key = 1001, 264, 0.5, 3, 0xABCDEF
    x = R.dyadic((rows, cols), 4, g, "cpu")
    R.assert_sum_exact(rows, 4 / (1 - rate))
    masked = R.drop32(x, rate, site, key)
    want = masked.double().sum(0)
    assert torch.equal(masked.sum(0, dtype=torch.float32).double(), want)      # exact in fp32 in any order
    assert not torch.equal(masked[:-1].double().sum(0), want)
    assert not torch.equal(x.double().sum(0), want)


def test_gelu_grad_and_pool_and_token_refs_are_autograd():
    x = torch.linspace(-8, 8, 4001, dtype=torch.float64).requires_grad_(True)
    R.gelu_tanh(x).sum().backward()
    grad, bound = R.gelu_tanh_grad(x.detach())
    assert (grad - x.grad).abs().max() < 1e-13
    assert (bound[x.detach().abs() < 1] < 2.0 ** -10).all()
    g = torch.Generator().manual_seed(6)
    B, T, D = 3, 17, 64
    x = torch.randn((B, T, D), generator=g, dtype=torch.float64)
    gamma = torch.randn(D, generator=g, dtype=torch.float64)
    dy = torch.randn((B, D), generator=g, dtype=torch.float64)
    for pool_mean in (0, 1):
        xr, gr = x.clone().requires_grad_(True), gamma.clone().requires_grad_(True)
        pooled = xr.mean(1) if pool_mean else xr[:, 0]
        (torch.nn.functional.layer_norm(pooled, (D,), gr, None, eps=1e-6) * dy).sum().backward()
        dp, dx, dg, db, _ = R.pool_ln_bwd(x, dy, gamma, pool_mean)
        assert (dx - xr.grad).abs().max() < 1e-12 and (dg - gr.grad).abs().max() < 1e-12
        assert torch.equal(dx[:, 0], dp)
    dpos, dcls, dbias = R.token_grads(x, 1)
    assert torch.equal(dcls, x[:, 0].sum(0)) and (dbias - x[:, 1:].sum((0, 1))).abs().max() < 1e-12
