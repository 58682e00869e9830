"""Time the decode half of the StyleGAN purifiers' input gradient: `from_codes` forward with tape + backward to the W+ codes.

    python scripts/bench_stylegan_grad.py [--mode bf16|fp32] [--steps K] [--warmup W] [--cases gender:32,gender:128,cars:64,cars:256]

One JSON line per case: ms per forward + backward, codes-gradients per second, peak HBM (torch allocator), and the share of the new
backward kernels (styled_bias_act_bwd, style_bwd, image_pool_out_bwd, latent_lerp_bwd) in a separate, CUDA-event-instrumented pass.
Weights are the seeded synthetic checkpoints of bench.py; codes are N(0, 1).  Every step runs > 1 GB of activations through the
126 MB L2, so no explicit flush is done.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

NEW_OPS = ("styled_bias_act_bwd", "style_bwd", "image_pool_out_bwd", "latent_lerp_bwd")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def step(dm, codes, g_logits):
    c = codes.detach().requires_grad_()
    logits = dm.from_codes(c)
    g, = torch.autograd.grad(logits, [c], g_logits)
    return g


def run_case(workload, batch, mode, steps, warmup):
    import bench
    from gen_adversarial_b200 import ops
    dev = torch.device("cuda:0")
    dm = bench.make_ours(workload, mode, dev)
    dm.noise_seed = 1234
    n_codes = dm.autoencoder.decoder.n_latent
    gen = torch.Generator().manual_seed(0)
    codes = torch.randn(batch, n_codes, 512, generator=gen).to(dev)
    g_logits = torch.randn(batch, dm.classifier.classifier.n_classes, generator=gen).to(dev)
    for _ in range(warmup):
        step(dm, codes, g_logits)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step(dm, codes, g_logits)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak_gb = torch.cuda.max_memory_allocated(dev) / 1e9
    # instrumented pass: every op bracketed by CUDA events (slower than the timed window; shares only)
    ops.TIMER, ops.TIME_ALL = ops.KernelTimer(), True
    try:
        step(dm, codes, g_logits)
        agg = ops.TIMER.summary()
    finally:
        ops.TIMER, ops.TIME_ALL = None, False
    total = sum(a["ms"] for a in agg.values())
    new = {name: sum(a["ms"] for k, a in agg.items() if k.split(" ")[0].split(":")[-1] == name) for name in NEW_OPS}
    del dm
    torch.cuda.empty_cache()
    return {"workload": workload, "mode": mode, "batch": batch, "steps": steps, "warmup": warmup, "ms_fwd_tape_bwd": ms,
            "codes_grads_per_s": batch * 1000.0 / ms, "hbm_peak_gb": round(peak_gb, 2),
            "instrumented_ms": total, "new_kernel_ms": new, "new_kernel_share": sum(new.values()) / total if total else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--cases", default="gender:32,gender:128,cars:64,cars:256")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stylegan_grad.py measures on a CUDA device; none is available")
    gpu = gpu_info()
    for case in args.cases.split(","):
        wl, b = case.split(":")
        try:
            r = run_case(wl, int(b), args.mode, args.steps, args.warmup)
        except torch.cuda.OutOfMemoryError as e:
            r = {"workload": wl, "batch": int(b), "mode": args.mode, "error": f"out of memory: {str(e).splitlines()[0]}"}
            torch.cuda.empty_cache()
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
