"""The on-device training step, phase by phase: train_forward, the cross-entropy kernel, backward, and
vitb200_adamw_step (global norm + AdamW update + in-place re-pack of the 16-bit weights).
    python profiles/run_train_step.py [--steps 20] [--out DIR]   (writes DIR/r04_train_step.md)

ViT-B/16 at batch 256 and ViT-L/16 at batch 128, fp16 and bf16.  Every step records a CUDA event between the phases;
the figures are medians over the timed steps after three warm-up steps.  The optimiser phase moves about 28 bytes per
parameter (read p, g, mu, nu; write p, mu, nu) plus the refresh, far more than the 126 MB L2, so it streams from HBM.
Once (ViT-B/16, fp16, batch 256) the step a user had to write before this existed is timed for comparison:
vjp_fn (every leaf gradient copied to the host), AdamW in numpy float32, and the weights uploaded and re-packed by
ViT.apply's engine cache.  The GPU's name, power limit and maximum SM clock are read in the same run."""
import os
import statistics
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "profiles"))
sys.path.insert(0, str(ROOT / "tests"))
from _util import C2, C3  # noqa: E402
from run_input_grad import gpu_info  # noqa: E402
from vit_flax_b200 import ViT, adamw, init_params, perturb_params  # noqa: E402
from vit_flax_b200.params import count_params  # noqa: E402

PHASES = ["train_forward", "xent", "backward", "adamw_step"]


def time_steps(cfg, batch, precision, steps):
    variables = perturb_params(init_params(seed=1, **cfg), seed=2)
    tr = ViT(**cfg).trainer(variables, adamw(1e-4, max_grad_norm=1.0), precision=precision, max_batch=batch)
    eng = tr._eng
    x = torch.randn((batch, 224, 224, 3), device="cuda")
    y = torch.randint(0, cfg["num_classes"], (batch,), device="cuda", dtype=torch.int32)
    logits = torch.empty((batch, cfg["num_classes"]), device="cuda")
    dl = torch.empty_like(logits)
    scale = 2.0 ** round(np.log2(batch))
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(PHASES) + 1)] for _ in range(steps + 3)]
    for s in range(steps + 3):
        e = ev[s]
        e[0].record()
        eng.train_forward(x, out=logits)
        e[1].record()
        eng.softmax_xent(logits, y, dscale=scale, dlogits=dl)
        e[2].record()
        eng.backward(dl)
        e[3].record()
        eng.adamw_step(lr=1e-4, b1=0.9, b2=0.999, eps=1e-8, weight_decay=1e-4, max_grad_norm=1.0, grad_scale=1.0 / scale)
        e[4].record()
    torch.cuda.synchronize()
    out = {}
    for i, name in enumerate(PHASES):
        out[name] = statistics.median(ev[s][i].elapsed_time(ev[s][i + 1]) for s in range(3, steps + 3))
    out["step"] = statistics.median(ev[s][0].elapsed_time(ev[s][-1]) for s in range(3, steps + 3))
    count, skipped, _ = tr.last_step()
    assert count == steps + 3 and skipped == 0
    n = count_params(**cfg)
    out["params_M"] = n / 1e6
    out["update_GBps"] = 28 * n / (out["adamw_step"] * 1e-3) / 1e9
    return out


def kernel_split(cfg, batch, precision, steps=5):
    """Device time of each kernel of vitb200_adamw_step, from torch.profiler in a run of its own (the profiler slows the
    host, so the phase timings above come from a separate, unprofiled run).  The optimiser's kernels are those from a
    sumsq_kernel up to the next step's patchify: the names alone do not say it, since the backward also casts."""
    from torch.profiler import ProfilerActivity, profile
    variables = perturb_params(init_params(seed=1, **cfg), seed=2)
    tr = ViT(**cfg).trainer(variables, adamw(1e-4, max_grad_norm=1.0), precision=precision, max_batch=batch)
    x = torch.randn((batch, 224, 224, 3), device="cuda")
    y = torch.randint(0, cfg["num_classes"], (batch,), device="cuda")
    for _ in range(3):
        tr.step(x, y)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps + 1):
            tr.step(x, y)
        torch.cuda.synchronize()
    kern = []
    for e in prof.profiler.kineto_results.events():
        if e.device_type() != torch.autograd.DeviceType.CUDA:
            continue
        start = e.start_ns() if hasattr(e, "start_ns") else e.start_us() * 1000
        dur = e.duration_ns() if hasattr(e, "duration_ns") else e.duration_us() * 1000
        kern.append((start, dur, e.name()))
    kern.sort()
    groups, spans, window = {}, [], None
    for start, dur, name in kern:
        if "sumsq_kernel" in name:
            window = []
        elif window is not None and "patchify" in name:       # the window closes: count it
            spans.append(max(s + d for s, d, _ in window) - window[0][0])
            for _, d, short in window:
                n, t = groups.get(short, (0, 0))
                groups[short] = (n + 1, t + d)
            window = None
        if window is not None:
            window.append((start, dur, name.split("(")[0].split("::")[-1].split("<")[0].replace("void ", "")))
    k = len(spans)
    assert k >= steps, f"found {k} optimiser windows"
    rows = sorted(((t / k / 1e3, n / k, name) for name, (n, t) in groups.items()), reverse=True)
    return statistics.median(s / 1e3 for s in spans), rows


def time_host_loop(cfg, batch, iters=2):
    """vjp -> host gradients -> numpy AdamW -> re-upload through ViT.apply's cache: one iteration per row."""
    from vit_flax_b200.params import flatten_params
    from vit_flax_b200.checkpoint import _unflatten
    v = ViT(**cfg)
    params = {k: np.array(a, np.float32) for k, a in flatten_params(perturb_params(init_params(seed=1, **cfg), seed=2)).items()}
    mu = {k: np.zeros_like(a) for k, a in params.items()}
    nu = {k: np.zeros_like(a) for k, a in params.items()}
    x = torch.randn((batch, 224, 224, 3), device="cuda")
    y = torch.randint(0, cfg["num_classes"], (batch,), device="cuda")
    times = []
    for t in range(1, iters + 2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        logits, vjp_fn = v.vjp({"params": _unflatten(params)}, x)
        p = torch.softmax(logits, 1)
        p[torch.arange(batch), y] -= 1
        grads = flatten_params(vjp_fn(p / batch))
        for k in params:      # optax.adamw arithmetic, numpy float32
            g = grads[k]
            mu[k] = 0.9 * mu[k] + 0.1 * g
            nu[k] = 0.999 * nu[k] + 0.001 * g * g
            params[k] = params[k] - 1e-4 * ((mu[k] / (1 - 0.9 ** t)) / (np.sqrt(nu[k] / (1 - 0.999 ** t)) + 1e-8)
                                            + 1e-4 * params[k])
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    return times[1:]   # the first iteration also builds the engine


def main():
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 20
    out_dir = Path(sys.argv[sys.argv.index("--out") + 1]) if "--out" in sys.argv else None
    info = gpu_info()
    lines = [f"GPU: {info['gpu']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}.", "",
             f"Medians over {steps} steps after 3 warm-up steps; ms per phase (CUDA events).", "",
             "| model | batch | operands | train_forward | xent | backward | adamw_step | step | params (M) | adamw_step GB/s at 28 B/param |",
             "|---|---|---|---|---|---|---|---|---|---|"]
    for name, cfg, batch in (("ViT-B/16", C2, 256), ("ViT-L/16", C3, 128)):
        for precision in ("fp16", "bf16"):
            r = time_steps(cfg, batch, precision, steps)
            lines.append(f"| {name} | {batch} | {precision} | {r['train_forward']:.2f} | {r['xent']:.3f} | {r['backward']:.2f} | "
                         f"{r['adamw_step']:.3f} | {r['step']:.2f} | {r['params_M']:.1f} | {r['update_GBps']:.0f} |")
            print(lines[-1], flush=True)
            torch.cuda.empty_cache()
    os.environ["VITB200_LN_FOLD"] = "0"   # no folded copies to refresh: what the fold costs the optimiser phase
    r = time_steps(C2, 256, "fp16", steps)
    del os.environ["VITB200_LN_FOLD"]
    lines.append(f"| ViT-B/16, LayerNorm fold off | 256 | fp16 | {r['train_forward']:.2f} | {r['xent']:.3f} | {r['backward']:.2f} | "
                 f"{r['adamw_step']:.3f} | {r['step']:.2f} | {r['params_M']:.1f} | {r['update_GBps']:.0f} |")
    print(lines[-1], flush=True)
    torch.cuda.empty_cache()
    span, rows = kernel_split(C2, 256, "fp16")
    busy = sum(r[0] for r in rows)
    lines += ["", "Kernels of `adamw_step`, ViT-B/16 fp16 batch 256 (torch.profiler, own run, per step): window "
              f"{span * 1e3:.0f} µs from the first to the last kernel's end, {busy * 1e3:.0f} µs of it in kernels.", "",
              "| kernel | launches | µs |", "|---|---|---|"]
    lines += [f"| `{name}` | {n:.0f} | {t * 1e3:.0f} |" for t, n, name in rows]
    print("\n".join(lines[-len(rows) - 4:]), flush=True)
    host = time_host_loop(C2, 256)
    lines += ["", "Host round-trip loop (ViT-B/16, fp16, batch 256: vjp + leaf gradients to the host + numpy AdamW + "
              f"re-upload and re-pack), ms per iteration: {', '.join(f'{t:.0f}' for t in host)}."]
    print(lines[-1])
    text = "# r04: the on-device training step, phase by phase\n\n" + \
        "Generated by `python profiles/run_train_step.py --steps 20 --out profiles`.\n\n" + "\n".join(lines) + "\n"
    if out_dir:
        out_dir.mkdir(parents=True, exist_ok=True)
        (out_dir / "r04_train_step.md").write_text(text)


if __name__ == "__main__":
    main()
