"""Backward pass by what it differentiates: wrt = params / input / both, plus the two kernels the image gradient adds.
    python profiles/run_input_grad.py [C2] [batch 256] [fp16|bf16] [rounds 20] [--out result.json]

One process, one engine: every round runs train_forward + backward once per mode, the modes in rotating order, and
times the backward alone with CUDA events after two warm-up rounds.  Then the patch-feature GEMM
(dpatches = dY W_patch^T through vitb200_gemm_tc, fp32 output) and unpatchify (vitb200_unpatchify) are timed on their
own at the same shapes, 50 back-to-back launches each.  Their working sets (155 MB of fp32 patch features + 154 MB of
image gradient at ViT-B/16 batch 256) exceed the 126 MB L2, so the launches stream from HBM.  The GPU's name,
power limit and maximum SM clock are read in the same run and printed with the numbers."""
import ctypes as C
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from _util import C2, C3, C4, C5  # noqa: E402
from vit_flax_b200 import _lib, init_params, perturb_params  # noqa: E402
from vit_flax_b200.engine import Engine  # noqa: E402

MODES = ["params", "input", "both"]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the timings stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"not read ({e})", "max_sm_clock": "not read"}


def time_launches(fn, n=50):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out in args:
        args.remove(out)
    name = args[0] if args else "C2"
    batch = int(args[1]) if len(args) > 1 else 256
    dtype = args[2] if len(args) > 2 else "fp16"
    rounds = int(args[3]) if len(args) > 3 else 20
    cfg = dict(C2=C2, C3=C3, C4=C4, C5=C5)[name]
    assert torch.cuda.is_available(), "this measurement needs the GPU"
    info = gpu_info()
    eng = Engine(precision=dtype, max_batch=batch, **cfg)
    eng.load_params(perturb_params(init_params(seed=1, **cfg), seed=2))
    s, ps = cfg["image_size"], cfg["patch_size"]
    x = torch.randn((batch, s, s, 3), device="cuda")
    logits = torch.empty((batch, cfg["num_classes"]), device="cuda")
    dl = torch.randn((batch, cfg["num_classes"]), device="cuda") / batch
    dimg = torch.empty_like(x)
    times = {m: [] for m in MODES}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds + 2):
        for k in range(len(MODES)):
            m = MODES[(r + k) % len(MODES)]
            eng.train_forward(x, out=logits)
            e0.record()
            eng.backward(dl, wrt=m, dimages=dimg if m != "params" else None)
            e1.record()
            torch.cuda.synchronize()
            if r >= 2:
                times[m].append(e0.elapsed_time(e1))
    # the image gradient is the same bits with and without the parameter gradients
    eng.train_forward(x, out=logits)
    a = eng.backward(dl, wrt="input").clone()
    b = eng.backward(dl, wrt="both").clone()
    same_dx = bool(torch.equal(a, b))
    eng.close()

    # the two new kernels on their own, at the model's shapes
    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    T = (s // ps) ** 2 + 1
    K0 = ps * ps * 3
    K0pad = -(-K0 // 64) * 64
    D, R = cfg["dim"], batch * T
    tdt, dt = (torch.float16, _lib.DT_F16) if dtype == "fp16" else (torch.bfloat16, _lib.DT_BF16)
    dy = torch.randn((R, D), device="cuda").to(tdt)
    wf = torch.zeros((K0pad, D), device="cuda", dtype=tdt)
    wf[:K0] = torch.randn((K0, D), device="cuda").to(tdt) / D ** 0.5
    zeros = torch.zeros(K0pad, device="cuda")
    dpatch = torch.empty((R, K0pad), device="cuda")
    gemm_ms = time_launches(lambda: _lib.check(lib.vitb200_gemm_tc(st, dy.data_ptr(), wf.data_ptr(), zeros.data_ptr(), dpatch.data_ptr(),
                                                                   R, K0pad, D, _lib.EPI_BIAS_F32, None, 0, dt)))
    unp_ms = time_launches(lambda: _lib.check(lib.vitb200_unpatchify(st, dpatch.data_ptr(), dimg.data_ptr(), batch, s, s, 3, ps, ps,
                                                                     K0pad, 0, 1)))
    gemm_flop = 2.0 * R * K0pad * D
    unp_bytes = 2.0 * batch * s * s * 3 * 4          # every patch feature read once, every pixel written once
    med = {m: statistics.median(v) for m, v in times.items()}
    res = dict(info, config=name, batch=batch, precision=dtype, rounds=rounds,
               backward_ms_median={m: round(v, 3) for m, v in med.items()},
               backward_ms_min={m: round(min(v), 3) for m, v in times.items()},
               backward_ms_max={m: round(max(v), 3) for m, v in times.items()},
               both_minus_params_ms=round(med["both"] - med["params"], 3),
               input_over_params=round(med["input"] / med["params"], 3),
               dx_input_equals_dx_both=same_dx,
               patch_dgrad_gemm=dict(M=R, N=K0pad, K=D, ms=round(gemm_ms, 4), gflop=round(gemm_flop / 1e9, 1),
                                     tflops=round(gemm_flop / gemm_ms / 1e9, 1)),
               unpatchify=dict(ms=round(unp_ms, 4), mbytes=round(unp_bytes / 1e6, 1), gbps=round(unp_bytes / unp_ms / 1e6, 0)))
    print(json.dumps(res, indent=1))
    if out:
        Path(out).parent.mkdir(parents=True, exist_ok=True)
        Path(out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
