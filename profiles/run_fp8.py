"""precision='fp8' against fp16 (and bf16) in one process, alternated:
    python profiles/run_fp8.py [--steps 20] [--out DIR]   (writes DIR/r05_fp8.md and DIR/r05_fp8.json)

ViT-B/16 at batch 256 and ViT-L/16 at batch 128.  Engines for fp16 (the default LayerNorm-fold schedule), fp16 on the
LayerNorm-kernel schedule (VITB200_LN_FOLD=0, the schedule fp8 runs), fp8 and bf16 share the same weights and images;
every round times `steps` forwards of each in turn with CUDA events (median per forward), after warm-up, so that clock
and neighbour drift hit all of them alike.  Separate profiled forwards (a CUDA event before every launch,
``Engine.profile_forward``) give the device time of to_qkv, FeedForward Dense_0 and Dense_1 (and to_out) per layer,
turned into TFLOP/s (torch.profiler's kernel records were tried for this and dropped a record of a 98-GEMM forward).
The images (256 x 224 x 224 x 3 fp32, 154 MB) and the activations exceed the 126 MB L2.  A parity block compares the
fp8 logits of 256 images with the fp32 oracle.  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "profiles"))
sys.path.insert(0, str(ROOT / "tests"))
from _util import C2, C3, images_for, oracle_logits  # noqa: E402
from run_input_grad import gpu_info  # noqa: E402
from vit_flax_b200 import init_params, perturb_params  # noqa: E402
from vit_flax_b200.engine import Engine  # noqa: E402

ARMS = ["fp16", "fp16-ln", "fp8", "bf16"]


def make_engine(arm, cfg, batch, variables):
    prec = arm.split("-")[0]
    old = os.environ.get("VITB200_LN_FOLD")
    if arm == "fp16-ln":
        os.environ["VITB200_LN_FOLD"] = "0"          # read when the handle is created
    try:
        eng = Engine(precision=prec, max_batch=batch, **cfg)
    finally:
        if old is None:
            os.environ.pop("VITB200_LN_FOLD", None)
        else:
            os.environ["VITB200_LN_FOLD"] = old
    eng.load_params(variables)
    return eng


def gemm_flops(cfg, batch):
    T = (cfg["image_size"] // cfg["patch_size"]) ** 2 + 1
    R, D, H, I = batch * T, cfg["dim"], cfg["mlp_dim"], cfg["heads"] * 64
    return {"qkv": 2 * R * D * 3 * I, "ff1": 2 * R * D * H, "ff2": 2 * R * H * D}


def per_gemm_ms(eng, x, out, depth, reps=5):
    """Per-launch device time of to_out / to_qkv / FF Dense_0 / FF Dense_1, mean per layer (ms), from the library's
    profiled forward (a CUDA event before every launch, vitb200_profile_forward), in runs of their own."""
    acc = {"qkv": [], "out": [], "ff1": [], "ff2": []}
    for _ in range(reps):
        cat = eng.profile_forward(x, out=out)
        for k in acc:
            ms, n = cat[f"gemm_{k}"]
            assert n == depth, f"{n} {k} launches for {depth} layers"
            acc[k].append(ms / n)
    return {k: statistics.median(v) for k, v in acc.items()}


def run(cfg, batch, steps, rounds, parity):
    variables = perturb_params(init_params(seed=1, **cfg), seed=2)
    img = images_for(cfg, batch, seed=0)
    x = torch.as_tensor(img, device="cuda")
    engines = {a: make_engine(a, cfg, batch, variables) for a in ARMS}
    outs = {a: torch.empty((batch, cfg["num_classes"]), device="cuda") for a in ARMS}
    for a in ARMS:                                   # warm-up: module load, tensor maps, first launches
        for _ in range(3):
            engines[a].forward(x, out=outs[a])
    torch.cuda.synchronize()
    times = {a: [] for a in ARMS}
    for _ in range(rounds):
        for a in ARMS:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            ev[0].record()
            for s in range(steps):
                engines[a].forward(x, out=outs[a])
                ev[s + 1].record()
            torch.cuda.synchronize()
            times[a] += [ev[s].elapsed_time(ev[s + 1]) for s in range(steps)]
    res = {"config": {k: cfg[k] for k in ("dim", "depth", "heads", "mlp_dim")}, "batch": batch,
           "forward_ms": {a: statistics.median(t) for a, t in times.items()},
           "forward_ms_spread": {a: [min(t), max(t)] for a, t in times.items()}}
    fl = gemm_flops(cfg, batch)
    res["gemm_ms"], res["gemm_tflops"] = {}, {}
    for a in ARMS:
        ms = per_gemm_ms(engines[a], x, outs[a], cfg["depth"])
        res["gemm_ms"][a] = ms
        res["gemm_tflops"][a] = {k: fl[k] / (ms[k] * 1e-3) / 1e12 for k in fl}
    if parity:
        y8 = outs["fp8"].cpu().numpy()
        y16 = outs["fp16"].cpu().numpy()
        want = np.concatenate([oracle_logits(variables, img[i:i + 32], cfg) for i in range(0, batch, 32)])
        res["parity"] = {"images": batch, "fp8_max_abs": float(np.abs(y8 - want).max()),
                         "fp8_rms": float(np.sqrt(((y8 - want) ** 2).mean())),
                         "fp16_max_abs": float(np.abs(y16 - want).max()),
                         "fp8_top1_agree": float((y8.argmax(1) == want.argmax(1)).mean()),
                         "fp16_top1_agree": float((y16.argmax(1) == want.argmax(1)).mean())}
    for e in engines.values():
        e.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=".", help="directory for r05_fp8.md / r05_fp8.json")
    a = ap.parse_args()
    info = gpu_info()
    results = [run(C2, 256, a.steps, a.rounds, True), run(C3, 128, a.steps, a.rounds, False)]
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "r05_fp8.json").write_text(json.dumps({"gpu": info, "results": results}, indent=1))
    lines = [f"GPU: {info['gpu']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}; "
             f"{a.rounds} alternated rounds x {a.steps} forwards per arm, medians.", ""]
    for r in results:
        lines.append(f"## dim {r['config']['dim']}, depth {r['config']['depth']}, batch {r['batch']}")
        lines.append("| arm | forward ms (min..max) | qkv ms / TFLOP/s | FF1 ms / TFLOP/s | FF2 ms / TFLOP/s | to_out ms |")
        lines.append("|---|---|---|---|---|---|")
        for arm in ARMS:
            g, t = r["gemm_ms"][arm], r["gemm_tflops"][arm]
            lo, hi = r["forward_ms_spread"][arm]
            lines.append(f"| {arm} | {r['forward_ms'][arm]:.2f} ({lo:.2f}..{hi:.2f}) | {g['qkv']:.3f} / {t['qkv']:.0f} | "
                         f"{g['ff1']:.3f} / {t['ff1']:.0f} | {g['ff2']:.3f} / {t['ff2']:.0f} | {g['out']:.3f} |")
        if "parity" in r:
            lines.append("")
            lines.append("parity vs the fp32 oracle: " + ", ".join(f"{k} {v:.4g}" for k, v in r["parity"].items()))
        lines.append("")
    (out / "r05_fp8.md").write_text("\n".join(lines))
    print("\n".join(lines))


if __name__ == "__main__":
    main()
