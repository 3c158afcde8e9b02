"""The fp8 emulation (tests/_fp8_oracle.py) against what pins it on the CPU: the oracle's own fp16 emulation, the E4M3
format's known values, and the accuracy floor that makes fp8 an opt-in precision with a derived tolerance."""
import numpy as np
import torch

from oracle import vit_torch
from vit_flax_b200.params import init_params, perturb_params
from _fp8_oracle import decode_e4m3, e4m3, e4m3_codes, quantize_weight, vit_forward_fp8
from _util import C2, TINY, TINY_MEAN, images_for


def test_emulation_with_fp16_rounding_is_the_oracle_fp16_forward():
    """With every E4M3 site rounded to fp16 instead (unit weight scales) the emulation is, bit for bit, the oracle's
    fp16 emulation of the LayerNorm-kernel schedule; with no rounding at all it is the fp32 oracle."""
    for cfg, pool in ((TINY, "cls"), (TINY_MEAN, "mean"), (dict(C2, depth=2), "cls")):
        v = perturb_params(init_params(seed=1, **cfg), seed=2)
        img = images_for(cfg, 3, seed=0)
        pt = vit_torch.tree_to_torch(v)
        want16 = vit_torch.vit_forward(pt, img, pool=pool, operand_dtype=torch.float16, **cfg).numpy()
        np.testing.assert_array_equal(vit_forward_fp8(v, img, pool=pool, rounding="fp16", **cfg), want16)
        want32 = vit_torch.vit_forward(pt, img, pool=pool, **cfg).numpy()
        np.testing.assert_allclose(vit_forward_fp8(v, img, pool=pool, rounding="none", **cfg), want32, rtol=0, atol=2e-5)


def test_e4m3_rounding_known_values():
    x = torch.tensor([0.0, 1.0, 1.0625, 1.1875, 448.0, 460.0, 1e6, -1e6, 2.0 ** -9, 2.0 ** -10, 3 * 2.0 ** -11, 240.0, 248.0])
    # 1.0625 is the midpoint of 1 and 1.125 -> even (1.0); 1.1875 -> 1.25 (even); saturation at 448; 2^-9 is the smallest
    # subnormal, 2^-10 ties to 0, 3 * 2^-11 rounds up to 2^-9; 248 is the midpoint of 240 and 256 -> 256 (even)
    want = [0.0, 1.0, 1.0, 1.25, 448.0, 448.0, 448.0, -448.0, 2.0 ** -9, 0.0, 2.0 ** -9, 240.0, 256.0]
    np.testing.assert_array_equal(e4m3(x).numpy(), np.array(want, np.float32))
    codes = np.arange(256, dtype=np.uint8)
    finite = codes[(codes & 0x7F) != 0x7F]                      # 0x7F / 0xFF are NaN in E4M3
    vals = decode_e4m3(finite)
    np.testing.assert_array_equal(e4m3_codes(vals.astype(np.float32))[vals != 0], finite[vals != 0])


def test_weight_quantisation_round_trips():
    rng = np.random.default_rng(0)
    W = (rng.standard_normal((200, 48)) * rng.uniform(0.01, 3.0, 48)).astype(np.float32)
    W[:, 5] = 0.0                                                # an all-zero column: scale 1, codes 0
    w8, s = quantize_weight(W)
    s = s.numpy()
    assert s[5] == 1.0 and np.all(w8[:, 5].numpy() == 0.0)
    amax = np.abs(W).max(0)
    nz = amax > 0
    np.testing.assert_array_equal(s[nz], (amax[nz] / np.float32(448.0)).astype(np.float32))
    assert np.abs(w8.numpy()).max() <= 448.0
    # every column's largest entry lands on (or right next to) the top code; the round trip is within half an E4M3 step
    back = w8.numpy() * s
    rel = np.abs(back - W) / np.maximum(np.abs(W), 2.0 ** -6 * s)
    assert rel.max() <= 2.0 ** -4 + 1e-6
    # exact E4M3 values times a power-of-two scale come back exactly
    exact = decode_e4m3(rng.integers(0, 0x7E, (64, 16), dtype=np.uint8)).astype(np.float32)
    exact[0] = 448.0
    w8b, sb = quantize_weight(exact * np.float32(0.25))
    np.testing.assert_array_equal(sb.numpy(), np.full(16, 0.25, np.float32))
    np.testing.assert_array_equal(w8b.numpy(), exact)


def test_fp8_operand_floor_on_vit_b16():
    """The setup of test_oracle.py::test_bf16_operand_floor_on_vit_b16: E4M3 on to_qkv / FF Dense_0 / FF Dense_1 moves
    unit-variance ViT-B/16 logits by about 0.32 (max-abs) from the fp32 oracle -- the 3-bit mantissa, not the range.
    fp8 is therefore an opt-in precision held to a bound derived from this emulation (tests/test_gpu_fp8.py)."""
    variables = perturb_params(init_params(seed=1, **C2), seed=2)
    img = images_for(C2, 8, seed=0)
    want = vit_torch.vit_forward(vit_torch.tree_to_torch(variables), img, **C2).numpy()
    got = vit_forward_fp8(variables, img, **C2)
    err = float(np.abs(got - want).max())
    rms = float(np.sqrt(((got - want) ** 2).mean()))
    print(f"[fp8 floor] ViT-B/16, 8 images: max-abs {err:.4f}, rms {rms:.4f}")
    assert 0.9 < want.std() < 1.1
    assert 0.2 < err < 0.5
