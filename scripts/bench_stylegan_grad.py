"""Time the decode half of the StyleGAN purifiers' input gradient: `from_codes` forward with tape + backward to the W+ codes.

    python scripts/bench_stylegan_grad.py [--mode bf16|fp32] [--steps K] [--warmup W] [--cases gender:32,gender:128,cars:64,cars:256]
    python scripts/bench_stylegan_grad.py --path images [--cases gender:32,gender:128]

--path images times the E4E encode half instead: `to_codes` forward with tape + backward to the images alone, and the whole chain
`from_codes(to_codes(x))` forward + backward to the images (image-gradients/s, peak HBM and the new kernels' share are of the chain).

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
NEW_OPS_IMAGES = ("phase_interleave", "subsample2x_bwd", "codes_assemble_bwd")


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


def step_images(dm, x, g, chain):
    xd = x.detach().requires_grad_()
    out = dm.from_codes(dm.to_codes(xd)) if chain else dm.to_codes(xd)
    gx, = torch.autograd.grad(out, [xd], g)
    return gx


def _timed_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _kernel_shares(fn, names):
    from gen_adversarial_b200 import ops
    ops.TIMER, ops.TIME_ALL = ops.KernelTimer(), True
    try:
        fn()
        agg = ops.TIMER.summary()
    finally:
        ops.TIMER, ops.TIME_ALL = None, False
    total = sum(a["ms"] for a in agg.values())
    new = {name: sum(a["ms"] for k, a in agg.items() if k.split(" ")[0].split(":")[-1] == name) for name in names}
    return total, new


def run_images_case(workload, batch, mode, steps, warmup):
    import bench
    dev = torch.device("cuda:0")
    dm = bench.make_ours(workload, mode, dev)
    dm.noise_seed = 1234
    gen = torch.Generator().manual_seed(0)
    x = torch.rand(batch, 3, 256, 256, generator=gen).to(dev)
    n_codes = dm.autoencoder.decoder.n_latent
    g_codes = torch.randn(batch, n_codes, 512, generator=gen).to(dev)
    g_logits = torch.randn(batch, dm.classifier.classifier.n_classes, generator=gen).to(dev)
    ms_enc = _timed_ms(lambda: step_images(dm, x, g_codes, False), steps, warmup)
    torch.cuda.reset_peak_memory_stats(dev)
    ms_chain = _timed_ms(lambda: step_images(dm, x, g_logits, True), steps, warmup)
    peak_gb = torch.cuda.max_memory_allocated(dev) / 1e9
    total, new = _kernel_shares(lambda: step_images(dm, x, g_logits, True), NEW_OPS_IMAGES)
    del dm
    torch.cuda.empty_cache()
    return {"workload": workload, "path": "images", "mode": mode, "batch": batch, "steps": steps, "warmup": warmup,
            "ms_to_codes_tape_bwd": ms_enc, "ms_chain_fwd_bwd": ms_chain, "image_grads_per_s": batch * 1000.0 / ms_chain,
            "hbm_peak_gb": round(peak_gb, 2), "instrumented_ms": total, "new_kernel_ms": new,
            "new_kernel_share": sum(new.values()) / total if total else None}


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
    ap.add_argument("--cases", default=None, help="workload:batch,... (default gender:32,gender:128,cars:64,cars:256; images: gender only)")
    ap.add_argument("--path", default="codes", choices=["codes", "images"])
    args = ap.parse_args()
    cases = args.cases or ("gender:32,gender:128,cars:64,cars:256" if args.path == "codes" else "gender:32,gender:128")
    if not torch.cuda.is_available():
        raise SystemExit("bench_stylegan_grad.py measures on a CUDA device; none is available")
    gpu = gpu_info()
    for case in cases.split(","):
        wl, b = case.split(":")
        if args.path == "images" and wl != "gender":
            raise SystemExit("--path images: only the gender (E4E) encoder has an input-gradient backward")
        try:
            r = (run_images_case if args.path == "images" else run_case)(wl, int(b), args.mode, args.steps, args.warmup)
        except torch.cuda.OutOfMemoryError as e:
            r = {"workload": wl, "batch": int(b), "mode": args.mode, "error": f"out of memory: {str(e).splitlines()[0]}"}
            torch.cuda.empty_cache()
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
