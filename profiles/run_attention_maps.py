"""What recording attention maps costs:
    python profiles/run_attention_maps.py [--reps 7] [--out FILE]   (default profiles/r06_attention_maps.md)

1. Per recorded layer, at ViT-B/16 batch 256 (T = 197) and ViT-H/14 batch 256 (T = 257): the probabilities kernel alone
   (vitb200_attention_probs on a to_qkv-shaped buffer) and the attention kernel with and without its row log-sum-exp
   (vitb200_attention_tc_lse / vitb200_attention_tc), CUDA events over 20 launches, median of `reps` rounds.  The write
   floor of a layer is its maps' bytes, B h T^2 4, over two rates: 6530 GB/s (BASELINE.md, HBM copy) and the rate of
   torch's fill_ of a buffer of the same size measured in this run (write-only traffic, like the kernel's).
2. ViT-B/16 batch 256 forwards, alternated in one process: apply, a recording forward of all 12 layers and one of layer
   0 (Engine.forward_attn into preallocated maps), `reps` rounds of 20 forwards each in a rotating order, median per
   forward.
The GPU's name and power limit are read in the same run."""
import argparse
import ctypes as C
import statistics
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "profiles"))
sys.path.insert(0, str(ROOT / "tests"))
from _util import C2, C4, images_for  # noqa: E402
from run_input_grad import gpu_info  # noqa: E402
from vit_flax_b200 import _lib, init_params, perturb_params  # noqa: E402
from vit_flax_b200.engine import Engine  # noqa: E402

COPY_GBS = 6530.0   # BASELINE.md: HBM copy rate of this B200


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def per_launch_ms(fn, n=20):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def kernels(lib, name, cfg, batch, reps):
    T = (cfg["image_size"] // cfg["patch_size"]) ** 2 + 1
    h, dt = cfg["heads"], _lib.DT_F16
    qkv = (torch.randn((batch * T, 3 * h * 64), device="cuda") * 0.5).to(torch.float16)
    out = torch.empty((batch * T, h * 64), dtype=torch.float16, device="cuda")
    lse = torch.empty((batch * h, T), device="cuda")
    maps = torch.empty((batch, h, T, T), device="cuda")
    fill = torch.empty_like(maps)
    arms = {
        "attention": lambda: lib.vitb200_attention_tc(stream(), qkv.data_ptr(), out.data_ptr(), batch, T, h, dt),
        "attention+lse": lambda: lib.vitb200_attention_tc_lse(stream(), qkv.data_ptr(), out.data_ptr(), lse.data_ptr(),
                                                              batch, T, h, dt),
        "probs": lambda: lib.vitb200_attention_probs(stream(), qkv.data_ptr(), lse.data_ptr(), maps.data_ptr(), batch, T,
                                                     h, dt),
        "fill_": lambda: fill.fill_(0.0),
    }
    _lib.check(arms["attention+lse"]())
    t = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            t[k].append(per_launch_ms(fn))
    med = {k: statistics.median(v) for k, v in t.items()}
    nbytes = batch * h * T * T * 4
    row = dict(name=name, T=T, batch=batch, heads=h, gb=nbytes / 1e9, **{f"{k}_us": 1e3 * v for k, v in med.items()})
    row["added_us"] = row["probs_us"] + row["attention+lse_us"] - row["attention_us"]
    row["floor_copy_us"] = nbytes / (COPY_GBS * 1e9) * 1e6
    row["fill_gbs"] = nbytes / (med["fill_"] * 1e-3) / 1e9
    row["probs_gbs"] = nbytes / (med["probs"] * 1e-3) / 1e9
    return row


def forwards(cfg, batch, reps):
    variables = perturb_params(init_params(seed=1, **cfg), seed=2)
    eng = Engine(precision="fp16", max_batch=batch, **cfg)
    eng.load_params(variables)
    x = torch.as_tensor(images_for(cfg, batch, seed=3), device="cuda")
    T, h, depth = eng.tokens, cfg["heads"], cfg["depth"]
    logits = torch.empty((batch, cfg["num_classes"]), device="cuda")
    all_maps = torch.empty((batch, depth, h, T, T), device="cuda")
    one_map = torch.empty((batch, 1, h, T, T), device="cuda")
    arms = {
        "apply": lambda: eng.forward(x, out=logits),
        f"record all {depth} layers": lambda: eng.forward_attn(x, list(range(depth)), out=logits, maps=all_maps),
        "record layer 0": lambda: eng.forward_attn(x, [0], out=logits, maps=one_map),
    }
    for fn in arms.values():   # warm-up: module loads, tensor maps, the lse scratch
        fn()
    torch.cuda.synchronize()
    t = {k: [] for k in arms}
    names = list(arms)
    for r in range(reps):      # the order rotates every round: no arm always follows the write-bound one
        for k in names[r % 3:] + names[:r % 3]:
            t[k].append(per_launch_ms(arms[k], n=20))
    eng.close()
    return {k: statistics.median(v) for k, v in t.items()}, all_maps.numel() * 4 / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_attention_maps.md"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs the GPU"
    lib = _lib.load()
    info = gpu_info()
    rows = [kernels(lib, "ViT-B/16", C2, 256, a.reps), kernels(lib, "ViT-H/14", C4, 256, a.reps)]
    fwd, all_gb = forwards(C2, 256, a.reps)
    base = fwd["apply"]
    L = [f"# Attention maps: cost of recording (r06)", "",
         f"Measured on {info['gpu']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}; fp16; "
         f"median of {a.reps} alternated rounds.  `python profiles/run_attention_maps.py`.", "",
         "## Per recorded layer (batch 256)", "",
         "| model | T | maps / layer | attention | attention + lse | probs kernel | added per layer | floor at 6530 GB/s | "
         "fill_ of the same bytes | probs write rate |",
         "|---|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        L.append(f"| {r['name']} | {r['T']} | {r['gb']:.3f} GB | {r['attention_us']:.1f} us | {r['attention+lse_us']:.1f} us | "
                 f"{r['probs_us']:.1f} us | {r['added_us']:.1f} us | {r['floor_copy_us']:.1f} us | {r['fill__us']:.1f} us "
                 f"({r['fill_gbs']:.0f} GB/s) | {r['probs_gbs']:.0f} GB/s |")
    L += ["", "Added per layer = probs kernel + (attention with lse - attention without).", "",
          "## Forward, ViT-B/16 batch 256", "", "| forward | time | over apply |", "|---|---|---|"]
    for k, v in fwd.items():
        L.append(f"| {k} | {v:.2f} ms | {v - base:+.2f} ms ({(v / base - 1) * 100:+.1f} %) |")
    L += ["", f"Recording all layers writes {all_gb:.2f} GB of maps.", ""]
    text = "\n".join(L)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(text)
    print(text)


if __name__ == "__main__":
    main()
