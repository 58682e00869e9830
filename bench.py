#!/usr/bin/env python
"""bench.py -- headline benchmark of the purification hot path (BASELINE.json).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload purify|pgd|gender|cars] [--extras 0|1]
                  [--dump-outputs DIR]

"step" = one pass of the hot path over one batch of synthetic input:
  workload purify (default, BASELINE configs[1]): NVAE CelebA-64 "ids" + configs/ours_learned_blur_ids.yaml
      (blur on, eps 0) + VGG11 classifier, batch 512 per GPU, bf16 tensor-core path, random-init weights of the
      C32 architecture (SURVEY 8d), synthetic images.  metric = purified img/s.
  workload pgd (BASELINE configs[4]): PGD-Linf (eps 8/255, step 2/255, 50 steps) through purifier + classifier.
  workload gender / cars (BASELINE configs[2] / [3]): StyleGAN-E4E @1024 + ResNet-50, batch 128 / Style-Transformer @512 +
      ResNeXt-50, batch 256.

The JSON line (one, on stdout, rank 0):
  value   : whole-job img/s with inputs resident in HBM, device-timed (CUDA events around the K steps, NO per-launch events
            inside), max over ranks.
  e2e     : the same through the reference-facing API (`NVAEDefenseModel.__call__`) from pinned HOST buffers, with the
            H2D copy of the batch and the D2H read of the logits inside the timed region.
  roofline: collected in a SEPARATE instrumented pass after the timed region (every tensor-core conv launch bracketed by CUDA
            events on the launching stream): the tcgen05 implicit-GEMM conv kernel, FLOP-weighted over all its launches, against
            MEASURED_PEAKS.json; `roofline_other_kernels`: the fused decoder cell and the HBM-bound kernels (GB/s each).
  cpu_baseline: the reference's own modules (kind "reference", oracle/_ref/reference through oracle/ref_import.py) or, when the tree
            is absent, the oracle port (kind "port") on the host cores, bounded sample.
  extras (default workload only): `strong_scaling` (configs[1] at GLOBAL batch 512 = 512/N per GPU, CUDA-graph replay), `pgd`
            (configs[4], short run, at every N), and at N = 1 `gender`, `cars` (configs[2], [3]) and `incumbent_gpu` (the UNMODIFIED
            reference modules on cuda:0 -- fp32 as the reference runs them, and under bf16 autocast -- the bar the kernels must beat).
--impl reference: the reference's own CPU implementation of the path on the host cores, same config, bounded sample per step.
--dump-outputs DIR: after the timed steps, what the last timed step returned to its caller (logits; for pgd the success flags, L-inf
            distances and adversarial images) as DIR/<name>.npy in float32, at most 64 MB in all.  Inputs, weights and the noise seeds
            are seeded, so two builds run with the same arguments can be compared output for output.
Multi-GPU (torchrun): batch sharded data-parallel, no data-path collective; the only collective is one
all-reduce of the int64[3] accuracy counters (SURVEY 8e).  scaling = weak (fixed 512 images per GPU).
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

YAML = {   # /root/reference/configs/*.yaml, verbatim
    "purify": {"file": "ours_learned_blur_ids.yaml",
               "interpolation_alphas": [0.000, 0.000, 0.001, 0.136, 0.131, 0.206, 0.179, 0.305, 0.347, 0.349, 0.465, 0.528, 0.551,
                                        0.606, 0.681, 0.676, 0.834, 0.800, 0.938, 0.911, 1.000, 1.000, 1.000, 1.000],
               "alpha_attenuation": 0.7, "initial_noise_eps": 0.0, "gaussian_blur_input": True},
    "pgd": {"file": "ours_cosine_noise_ids.yaml",
            "interpolation_alphas": [0.00, 0.02, 0.04, 0.07, 0.10, 0.15, 0.20, 0.25, 0.31, 0.37, 0.43, 0.50, 0.57, 0.63, 0.69,
                                     0.75, 0.80, 0.85, 0.90, 0.93, 0.96, 0.98, 1.00, 1.00],
            "alpha_attenuation": 0.7, "initial_noise_eps": 2.0, "gaussian_blur_input": False},
    "gender": {"file": "ours_linear_noise_gender.yaml",
               "interpolation_alphas": [0.05, 0.11, 0.16, 0.22, 0.27, 0.33, 0.38, 0.44, 0.50, 0.55, 0.61, 0.66, 0.72, 0.77, 0.83, 0.88, 0.94, 1.00],
               "alpha_attenuation": 1.0, "initial_noise_eps": 4.0, "gaussian_blur_input": False},
    "cars": {"file": "ours_cosine_blur_cars.yaml",
             "interpolation_alphas": [0.010, 0.038, 0.084, 0.146, 0.222, 0.309, 0.402, 0.500, 0.598, 0.691, 0.778, 0.854, 0.916, 0.962, 0.990, 1.000],
             "alpha_attenuation": 0.7, "initial_noise_eps": 0.0, "gaussian_blur_input": True},
}
LEARNED_BLUR_IDS, COSINE_NOISE_IDS = YAML["purify"], YAML["pgd"]
DEFAULT_BATCH = {"purify": 1024, "pgd": 1024, "gender": 128, "cars": 256}
RESOLUTION = {"purify": (3, 64, 64), "pgd": (3, 64, 64), "gender": (3, 256, 256), "cars": (3, 128, 128)}
N_CLASSES = {"purify": 100, "pgd": 100, "gender": 2, "cars": 4}
WORKLOAD_TEXT = {
    "purify": "BASELINE configs[1]: NVAE-C32 CelebA-64 ids purification (ours_learned_blur_ids.yaml: blur, eps 0, learned alphas x0.7) + "
              "VGG11 classifier, random-init weights",
    "pgd": "BASELINE configs[4]: PGD-Linf eps 8/255, step 2/255, %d steps (fwd + input-gradient each) + 1 eval forward, through NVAE-C32 "
           "purifier (ours_cosine_noise_ids.yaml) + VGG11, random-init weights",
    "gender": "BASELINE configs[2]: StyleGAN-E4E CelebA-HQ 256 gender (IR-SE50 + 18 map2style heads -> StyleGAN2 @1024 -> face_pool) "
              "ours_linear_noise_gender.yaml (eps 4, linear alphas) + ResNet-50, random-init weights",
    "cars": "BASELINE configs[3]: Style-Transformer Stanford Cars 128 (IR-SE50 + 3 transformer decoder layers -> StyleGAN2 @512) "
            "ours_cosine_blur_cars.yaml (blur, cosine alphas x0.7) + ResNeXt-50, random-init weights",
}
# algorithmic work (SURVEY 8d, unpruned, conv/linear MACs x2): ids = purifier 15.31 + VGG11 2.49 GFLOP per image
GFLOP_PER_IMAGE_FWD = {"purify": 17.8, "pgd": 17.8, "gender": 304.0, "cars": 172.0}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------- the reference's own modules
def reference_kind():
    from oracle import ref_import
    return "reference" if ref_import.reference_available() else "port"


def reference_cpu_callable(workload, sample):
    """-> (step() running the reference path once on `sample` images on the host cores, kind, description)"""
    from oracle import ref_import
    from gen_adversarial_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = YAML[workload]
    if ref_import.reference_available():
        dm, res, n_cls, _ = ref_import.build_reference_defense(workload, "cpu")
        x, _ = synth.synthetic_batch(sample, res, n_cls, seed=42)

        def step():
            with torch.no_grad():
                return dm(x)           # MLVGMDefenseModel.__call__ (abstract_models.py:161-193): fresh noise on every call
        return step, "reference", (f"UNMODIFIED reference modules (src/defenses/ours/models.py via oracle/ref_import.py, tree "
                                   f"{os.path.relpath(ref_import.REFERENCE_ROOT, ROOT) if ref_import.REFERENCE_ROOT.startswith(ROOT) else ref_import.REFERENCE_ROOT}), "
                                   f"torch CPU fp32, {cores} threads")
    if workload not in ("purify", "pgd"):
        raise RuntimeError("the reference tree is absent and the oracle port is wired for the NVAE workloads only")
    from oracle import nvae_ref
    from gen_adversarial_b200.nvae_spec import NvaeSpec, NVAE_C32_CONFIG, NVAE_C32_RESOLUTION
    spec = NvaeSpec(NVAE_C32_CONFIG, NVAE_C32_RESOLUTION)
    sd = synth.make_nvae_state_dict(seed=0)
    vgg = nvae_ref.build_vgg11(synth.make_vgg11_state_dict(100, seed=1), 100)
    x, _ = synth.synthetic_batch(sample, seed=42)
    alphas = [a * cfg["alpha_attenuation"] for a in cfg["interpolation_alphas"]]

    def step():
        g = torch.Generator().manual_seed(int(time.time() * 1e3) % (2 ** 31))
        noises = [torch.randn(s, generator=g) for s in spec.noise_shapes(sample)]
        with torch.no_grad():
            logits, _ = nvae_ref.defense_call(sd, spec, vgg, x, alphas, noises, cfg["initial_noise_eps"], cfg["gaussian_blur_input"])
        return logits
    return step, "port", f"oracle/nvae_ref.py (CPU restatement of the reference path), torch CPU fp32, {cores} threads"


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    wl = args.workload
    sample = args.ref_batch if args.ref_batch else {"purify": 64, "pgd": 64, "gender": 2, "cars": 2}[wl]
    step, kind, desc = reference_cpu_callable("purify" if wl == "pgd" else wl, sample)
    cores = os.cpu_count() or 1
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = sample * args.steps / dt
    line = {"impl": "reference", "metric": "purified_img_per_s", "value": val, "unit": "img/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_TEXT["purify" if wl == "pgd" else wl] + " -- " + desc,
                       "sample_batch": sample, "batch_per_gpu": sample, "global_batch": sample},
            "cpu_baseline": {"value": val, "unit": "img/s", "cores": cores, "kind": kind,
                             "sample": f"{args.steps} steps x batch {sample} of the same workload ({desc})"},
            "e2e": {"value": val, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=JSON_OUT or sys.stdout, flush=True)


def cpu_baseline(sample_batch=16, runs=2):
    step, kind, desc = reference_cpu_callable("purify", sample_batch)
    times = []
    for _ in range(runs + 1):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    t = statistics.median(times[1:])
    return {"value": sample_batch / t, "unit": "img/s", "cores": os.cpu_count() or 1, "kind": kind,
            "sample": f"batch {sample_batch}, 1 warm-up + median of {runs} calls of the same workload ({desc})"}


def incumbent_gpu(dev, workloads=("purify", "gender", "cars"), ours=None):
    """The UNMODIFIED reference modules on cuda:0 (SURVEY 8d 'reference-on-B200'): torch/cuDNN convs and the reference's own JIT-built
    upfirdn2d / fused_bias_act kernels -- the incumbent the hand-written path has to beat.  Two settings: fp32 exactly as the reference
    runs (torch defaults: cuDNN may use TF32 for convs, matmuls fp32) with cudnn.benchmark on, and the same modules under bf16 autocast.
    Batch = the BASELINE batch when it fits (the reference materialises per-sample modulated weights and 1024x1024 activations:
    StyleGAN workloads run at a smaller batch, stated).  img/s, CUDA events, 1 warm-up + 3 timed calls."""
    from oracle import ref_import
    from gen_adversarial_b200 import synth
    out = {}
    if not ref_import.reference_available():
        return {"unavailable": "reference tree absent (set GA_REFERENCE_ROOT or run oracle/build_ref.sh)"}
    torch.backends.cudnn.benchmark = True
    for wl in workloads:
        try:
            t0 = time.perf_counter()
            dm, res, n_cls, _ = ref_import.build_reference_defense(wl, str(dev))
            B = {"purify": 512, "gender": 16, "cars": 32}[wl]
            x, _ = synth.synthetic_batch(B, res, n_cls, seed=42)
            x = x.to(dev)
            entry = {"batch": B, "build_s": round(time.perf_counter() - t0, 1)}
            for tag, ctx in (("fp32_torch_defaults", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
                try:
                    def call():
                        with torch.no_grad():
                            if ctx is None:
                                return dm(x)
                            with ctx:
                                return dm(x)
                    call(); call()
                    torch.cuda.synchronize(dev)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(3):
                        call()
                    e1.record()
                    torch.cuda.synchronize(dev)
                    entry[tag] = {"img_per_s": 3 * B / (e0.elapsed_time(e1) / 1e3), "ms_per_call": e0.elapsed_time(e1) / 3}
                except Exception as ex:   # e.g. an op of the reference without a bf16 kernel
                    entry[tag] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
            if ours and wl in ours:
                entry["ours_img_per_s"] = ours[wl]
                best = max((v["img_per_s"] for v in entry.values() if isinstance(v, dict) and "img_per_s" in v), default=None)
                entry["ours_over_best_incumbent"] = ours[wl] / best if best else None
            out[wl] = entry
            del dm, x
            torch.cuda.empty_cache()
        except Exception as ex:
            out[wl] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
    out["note"] = ("reference = unmodified src/defenses/ours/models.py classes on cuda:0 through oracle/ref_import.py (3 import shims + kornia "
                   "restatement); same seeded synthetic checkpoints as the CUDA path; cudnn.benchmark=True")
    return out


# ----------------------------------------------------------------------------------------------- our arm (GPU)
def make_ours(workload, mode, dev, chunk=0):
    from gen_adversarial_b200 import synth
    from gen_adversarial_b200.defenses.ours.models import NVAEDefenseModel, CelebaIdentityClassifier
    cfg = YAML[workload]
    if workload == "gender":
        from gen_adversarial_b200.defenses.ours.models import E4EStyleGanDefenseModel, CelebaGenderClassifier
        clf = CelebaGenderClassifier(synth.make_resnet50_checkpoint(), dev, mode=mode)
        dm = E4EStyleGanDefenseModel(clf, synth.make_e4e_checkpoint(1024), cfg["interpolation_alphas"], cfg["alpha_attenuation"],
                                     cfg["initial_noise_eps"], cfg["gaussian_blur_input"], dev, mode=mode).eval()
    elif workload == "cars":
        from gen_adversarial_b200.defenses.ours.models import TransStyleGanDefenseModel, CarsTypeClassifier
        clf = CarsTypeClassifier(synth.make_resnext50_checkpoint(), dev, mode=mode)
        dm = TransStyleGanDefenseModel(clf, synth.make_trans_checkpoint(512), cfg["interpolation_alphas"], cfg["alpha_attenuation"],
                                       cfg["initial_noise_eps"], cfg["gaussian_blur_input"], dev, mode=mode).eval()
    else:
        nv = synth.make_nvae_checkpoint(seed=0)
        vg = {"state_dict": synth.make_vgg11_state_dict(100, seed=1, device=str(dev))}
        clf = CelebaIdentityClassifier(vg, dev, mode=mode)
        del vg
        dm = NVAEDefenseModel(clf, nv, cfg["interpolation_alphas"], cfg["alpha_attenuation"], cfg["initial_noise_eps"],
                              cfg["gaussian_blur_input"], dev, mode=mode).eval()
    if chunk and workload in ("gender", "cars"):
        dm.max_chunk = chunk
    return dm


class Ctx:
    """process-wide state of one bench run"""

    def __init__(self):
        self.rank, self.world, self.local = dist_env()
        self.dev = torch.device("cuda", self.local)
        self.dist = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = torch.tensor([v], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def measure(ctx, dm, workload, B, steps, warmup, mode, use_graph, pgd_steps=50, sample_clocks=False, global_offset=None,
            keep_outputs=False):
    """resident + end-to-end timing of one workload -> dict (identical on every rank); keep_outputs: "_outputs" holds host copies of
    what the last resident timed step returned"""
    from gen_adversarial_b200 import ops, synth, graphs as ga_graphs
    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    pgd = workload == "pgd"
    res, n_cls = RESOLUTION[workload], N_CLASSES[workload]
    dm.sample_offset = (rank * B) if global_offset is None else global_offset     # Philox streams keyed by the GLOBAL sample index
    dm.enable_cuda_graph(bool(use_graph))
    x_cpu, y_cpu = synth.synthetic_batch(B, res, n_cls, seed=42 + rank)
    x_host = x_cpu.pin_memory()
    x_dev = x_host.to(dev)
    y_dev = y_cpu.to(dev)
    counters = torch.zeros(3, dtype=torch.int64, device=dev)       # n_total, n_clean_correct, n_robust_correct
    logits_host = torch.empty((B, n_cls), dtype=torch.float32).pin_memory()
    if pgd:
        from gen_adversarial_b200.attacks import PGDLinf
        attack = PGDLinf(8 / 255, 2 / 255, pgd_steps)
        with torch.no_grad():
            y_dev = dm(x_dev).argmax(dim=1).clone()          # attack the model's own clean predictions (labels are synthetic)
        succ_host = torch.empty((B,), dtype=torch.bool).pin_memory()

    def step_resident():
        if pgd:
            succ, linf, adv = attack(x_dev, y_dev, dm)
            counters[2] += (~succ).sum()
            return {"success": succ, "linf": linf, "x_adv": adv}
        with torch.no_grad():
            logits = dm(x_dev)
        ops.softmax_xent(logits, y_dev, want_grad=False, counter=counters[1:2].view(torch.int64))
        return {"logits": logits}

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True)
        if pgd:
            succ, _, _ = attack(xd, y_dev, dm)
            succ_host.copy_(succ, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return succ
        with torch.no_grad():
            logits = dm(xd)
        logits_host.copy_(logits, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return logits

    # ---------------- resident timing: NO per-launch instrumentation inside
    ops.TIMER = None
    for _ in range(warmup):
        step_resident()
    ctx.barrier()
    counters.zero_()
    ops.launch_count(reset=True)
    replayed0 = ga_graphs.REPLAYED_LAUNCHES[0]
    torch.cuda.reset_peak_memory_stats(dev)
    sampler = ClockSampler(ctx.local) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step_resident()
    e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    # copied before the next call: a replayed CUDA graph returns static buffers that the next call overwrites
    outputs = {k: v.detach().to(torch.float32).cpu() for k, v in out.items()} if keep_outputs else None
    clocks = sampler.stop() if sampler else None
    launches = ops.launch_count(reset=True) + ga_graphs.REPLAYED_LAUNCHES[0] - replayed0      # eager launches + graph-replayed kernel nodes
    counters[0] = B * steps
    if world > 1:
        ctx.dist.all_reduce(counters, op=ctx.dist.ReduceOp.SUM)       # the path's only collective (24 bytes)
    value = world * B * steps / (ms / 1e3)

    # ---------------- end-to-end timing (host buffers, copies inside the timed region)
    for _ in range(max(1, warmup // 2)):
        step_e2e()
    ctx.barrier()
    e0.record()
    for _ in range(steps):
        step_e2e()
    e1.record()
    ctx.barrier()
    ms_e2e = ctx.max_over_ranks(e0.elapsed_time(e1))
    e2e_val = world * B * steps / (ms_e2e / 1e3)
    gflop = GFLOP_PER_IMAGE_FWD[workload] * ((2 * pgd_steps + 1) if pgd else 1)
    return {"value": value, "ms_per_step": ms / steps, "steps": steps, "warmup": warmup, "batch_per_gpu": B, "global_batch": B * world,
            "e2e": {"value": e2e_val, "unit": "img/s", "h2d_bytes_per_step": x_host.numel() * 4 * world,
                    "d2h_bytes_per_step": (B if pgd else logits_host.numel() * 4) * world},
            "gpu_launches": int(launches), "hbm_peak_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2), "clocks": clocks,
            "cuda_graph": bool(use_graph), "gflop_per_image_algorithmic": gflop, "tflops_algorithmic": value * gflop / 1e3,
            "counters": {"n_total": int(counters[0].item()), "n_clean_correct": int(counters[1].item()),
                         "n_robust_correct": int(counters[2].item())},
            "_x_dev": x_dev, "_y_dev": y_dev, "_outputs": outputs}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, outputs, rank, world):
    """outputs {name: host tensor, batch first} -> path/<name>.npy in float32 (name_rank<r>.npy on a multi-GPU run).  Above
    DUMP_LIMIT_BYTES in all (over the ranks), every array keeps the same seeded sample of batch rows, listed in sample_rows.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    budget = DUMP_LIMIT_BYTES // world - 4096                        # room for the .npy headers
    n = next(iter(outputs.values())).shape[0]
    row_bytes = sum(v[0].numel() * 4 for v in outputs.values())
    if n * row_bytes > budget:
        keep = budget // (row_bytes + 8)                             # + 8: the float64 row index
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        outputs = {k: v[rows] for k, v in outputs.items()}
        outputs["sample_rows"] = rows.to(torch.float64)
    suffix = f"_rank{rank}" if world > 1 else ""
    for k, v in outputs.items():
        np.save(os.path.join(path, f"{k}{suffix}.npy"), v.numpy())
    log(f"[bench] outputs of the last timed step -> {path}: " + ", ".join(f"{k}{tuple(v.shape)}" for k, v in outputs.items()))


def instrumented_pass(ctx, dm, workload, x_dev, y_dev, steps, step_ms, breakdown=False):
    """SEPARATE pass after the timed region: every tensor-core conv / fused-cell / HBM-bound launch bracketed by CUDA events on the
    launching stream -> (roofline, roofline_other_kernels).  The events cost ~2% of the step; `value` does not carry them."""
    from gen_adversarial_b200 import ops
    pk = peaks()
    dm.enable_cuda_graph(False)
    B = x_dev.shape[0]
    if workload == "pgd":
        dm.loss_input_grad(x_dev, y_dev)               # un-timed eager warm-up: the timed region replayed a graph (private memory pool);
        torch.cuda.synchronize()                       # the first eager iteration pays the allocator's cudaMallocs
    timer = ops.KernelTimer()
    ops.TIMER, ops.TIME_ALL = timer, True
    try:
        for _ in range(steps):
            if workload == "pgd":
                dm.loss_input_grad(x_dev, y_dev)           # ONE eager iteration of the attack: taping forward + dgrad sweep
            else:
                with torch.no_grad():
                    dm(x_dev)
    finally:
        ops.TIMER, ops.TIME_ALL = None, False
    agg_all = timer.summary()
    for a in agg_all.values():          # per-step figures
        for k in ("launches", "ms", "flops", "bytes"):
            a[k] = a[k] / steps
    if breakdown:
        rows = sorted(agg_all.items(), key=lambda kv: -kv[1]["ms"])
        log(f"{'op / shape':70s} {'n':>6s} {'ms/step':>9s} {'us/launch':>10s}")
        for k, a in rows[:70]:
            log(f"{k[:70]:70s} {a['launches']:6.0f} {a['ms']:9.3f} {1e3 * a['ms'] / a['launches']:10.1f}")
        log(f"sum of bracketed ops: {sum(a['ms'] for a in agg_all.values()):.2f} ms/step; uninstrumented step {step_ms:.2f} ms")
    conv = {k: a for k, a in agg_all.items() if not k.startswith(("op:", "fused:", "hbm:"))}
    fused = {k: a for k, a in agg_all.items() if k.startswith("fused:")}
    hbm = {k: a for k, a in agg_all.items() if k.startswith("hbm:")}
    tot_ms = sum(a["ms"] for a in conv.values())
    tot_fl = sum(a["flops"] for a in conv.values())
    ach = tot_fl / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
    top = sorted(conv.items(), key=lambda kv: -kv[1]["ms"])[:10]
    roof = {"bound": "tensor", "kernel": "conv3x3_tc_kernel + conv_tc_kernel (tcgen05 implicit-GEMM convs, all shapes, FLOP-weighted)",
            "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"],
            "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({pk['src']})",
            "traffic": 90.1e6, "traffic_unit": "bytes per launch",
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of the dominant shape (3x3, 64 -> 64 channels at 32x32, 512-image part-batch: "
                            "67.3 + 22.8 MB against 134.3 MB algorithmic x + W + y -- the previous kernel's output is partly still in L2) from the committed "
                            "ncu --set full capture profiles/r02_ncu_full_kernels_v1.md; `achieved` is FLOP-weighted over ALL conv shapes",
            "launches_per_step": round(sum(a["launches"] for a in conv.values())), "share_of_step": tot_ms / step_ms if step_ms > 0 else None,
            "collected": f"separate instrumented pass of {steps} step(s), per-launch CUDA events on the launching stream",
            "by_shape": [{"shape": k, "launches": round(a["launches"]), "ms": round(a["ms"], 3),
                          "tflops": round(a["flops"] / (a["ms"] * 1e-3) / 1e12, 1) if a["ms"] > 0 else None,
                          "gbs": round(a["bytes"] / (a["ms"] * 1e-3) / 1e9, 1) if a["ms"] > 0 else None} for k, a in top]}
    extra = []
    if fused:
        f_ms = sum(a["ms"] for a in fused.values()); f_fl = sum(a["flops"] for a in fused.values())
        # the SIMT stage of this kernel runs on the fp32 pipe: per hidden element 25 depthwise FMAs + ~5 FMA-pipe ops of the two SiLUs;
        # B200: 128 fp32 FMA lanes / clk / SM (scripts/ubench_pipes.cu: FFMA 1.0, FFMA2 0.5 warp-instructions / clk / SMSP)
        simt_ops = 0.0
        for k, a in fused.items():
            m_ = re.search(r"hw(\d+) c(\d+) hidden(\d+)", k)
            simt_ops += a["launches"] * B * int(m_.group(1)) ** 2 * int(m_.group(3)) * 30.0
        fp32_peak = 148 * 128 * 1965.0e6
        extra.append({"kernel": "mbconv_fused_kernel (decoder cell: expand 1x1 -> SiLU -> depthwise 5x5 -> SiLU -> project 1x1, hidden tensor on chip)",
                      "bound": "tensor", "achieved": f_fl / (f_ms * 1e-3) / 1e12, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                      "frac": f_fl / (f_ms * 1e-3) / 1e12 / pk["tf_sustained"], "launches_per_step": round(sum(a["launches"] for a in fused.values())),
                      "share_of_step": f_ms / step_ms if step_ms > 0 else None,
                      "fp32_pipe": {"achieved_tfma_s": simt_ops / (f_ms * 1e-3) / 1e12, "peak_tfma_s": fp32_peak / 1e12,
                                    "frac": simt_ops / (f_ms * 1e-3) / fp32_peak},
                      "by_shape": [{"shape": k[6:], "launches": round(a["launches"]), "us_per_launch": round(1e3 * a["ms"] / a["launches"], 1),
                                    "tflops": round(a["flops"] / (a["ms"] * 1e-3) / 1e12, 1)} for k, a in sorted(fused.items(), key=lambda kv: -kv[1]["ms"])]})
    # HBM-bound kernels: one entry per kernel class (algorithmic bytes of SURVEY 8d over the event time of its launches in the step)
    classes = {}
    for k, a in hbm.items():
        classes.setdefault(k[4:].split(" ")[0], {})[k[4:]] = a
    for name, shapes in sorted(classes.items(), key=lambda kv: -sum(a["ms"] for a in kv[1].values())):
        h_ms = sum(a["ms"] for a in shapes.values()); h_by = sum(a["bytes"] for a in shapes.values())
        if h_ms <= 0:
            continue
        extra.append({"kernel": name, "bound": "hbm", "achieved": h_by / (h_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                      "frac": h_by / (h_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "launches_per_step": round(sum(a["launches"] for a in shapes.values())),
                      "share_of_step": h_ms / step_ms if step_ms > 0 else None,
                      "by_shape": [{"shape": k, "launches": round(a["launches"]), "us_per_launch": round(1e3 * a["ms"] / a["launches"], 1),
                                    "gbs": round(a["bytes"] / (a["ms"] * 1e-3) / 1e9, 1)} for k, a in sorted(shapes.items(), key=lambda kv: -kv[1]["ms"])[:4]]})
    return roof, extra


def public(m):
    return {k: v for k, v in m.items() if not k.startswith("_")}


def run_ours(args):
    ctx = Ctx()
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    assert torch.cuda.is_available(), "bench.py (impl ours) needs a GPU: the product has no CPU path"
    torch.cuda.set_device(ctx.local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout to the ONE JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)
        ctx.dist = dist
    from gen_adversarial_b200.nvae_spec import NVAE_C32_CONFIG

    mode, wl = args.mode, args.workload
    sg = wl in ("gender", "cars")
    pgd = wl == "pgd"
    B = args.batch if args.batch is not None else DEFAULT_BATCH[wl]
    use_graph = (args.cuda_graph == 1) or (args.cuda_graph < 0 and (pgd or wl == "purify"))
    t_start = time.perf_counter()
    # every call draws its Philox noise seed from torch's CPU generator, which torch seeds at random in each process: a fixed seed
    # makes two runs with the same arguments compute the same outputs
    torch.manual_seed(0)
    dm = make_ours(wl, mode, dev, args.chunk)
    n_streams = args.streams if args.streams > 0 else (2 if wl in ("purify", "pgd") else 1)
    dm.set_streams(n_streams)              # public API: no-grad calls run as part-batches on CUDA streams (results unchanged)
    main = measure(ctx, dm, wl, B, args.steps, args.warmup, mode, use_graph and not sg, args.pgd_steps, sample_clocks=True,
                   keep_outputs=bool(args.dump_outputs))
    log(f"[bench] {wl}: {main['value']:.1f} img/s resident, {main['e2e']['value']:.1f} e2e ({time.perf_counter() - t_start:.0f} s)")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, main.pop("_outputs"), rank, world)
    roof, extra = None, []
    if not sg or args.breakdown:
        dm.set_streams(1)                  # per-launch events: one stream, so a launch's duration is its own
        roof, extra = instrumented_pass(ctx, dm, wl, main["_x_dev"] if not pgd else main["_x_dev"][:min(B, 512)],
                                        main["_y_dev"] if not pgd else main["_y_dev"][:min(B, 512)],
                                        1 if pgd else 2, main["ms_per_step"] if not pgd else 0.0, args.breakdown)
        dm.set_streams(n_streams)
        if n_streams > 1 and not pgd:
            roof["collected"] += f" with ONE stream; the timed region runs {n_streams} part-batches on {n_streams} streams, so shares add up to more than 1"
        if pgd:
            roof["share_of_step"] = None
            roof["collected"] += " (ONE eager attack iteration at batch <= 512: taping forward + dgrad sweep; the timed region replays a CUDA graph)"
    extras = {}
    if args.extras and wl == "purify":
        # ---- strong scaling of configs[1]: GLOBAL batch 512 split over the ranks, whole call replayed as a CUDA graph
        try:
            bs = max(1, 512 // world)
            m = measure(ctx, dm, "purify", bs, max(10, args.steps), 3, mode, True, global_offset=rank * bs)
            extras["strong_scaling"] = dict(public(m), scaling="strong", note="BASELINE configs[1] at GLOBAL batch 512 (512/N images per GPU), "
                                            "CUDA-graph replay of the whole call (public API: enable_cuda_graph)")
            log(f"[bench] strong scaling (global batch 512, {bs}/GPU): {m['value']:.1f} img/s")
        except Exception as ex:
            extras["strong_scaling"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
        del dm
        main.pop("_x_dev"), main.pop("_y_dev")
        torch.cuda.empty_cache()
        # ---- configs[4]: PGD-Linf, short run (1 attack of 50 iterations per rank), CUDA-graph replay of one iteration
        try:
            dmp = make_ours("pgd", mode, dev)
            dmp.set_streams(n_streams)
            m = measure(ctx, dmp, "pgd", args.pgd_batch, 1, 1, mode, True, args.pgd_steps)
            r_pgd, _ = instrumented_pass(ctx, dmp, "pgd", m["_x_dev"][:min(args.pgd_batch, 512)], m["_y_dev"][:min(args.pgd_batch, 512)], 1, 0.0)
            r_pgd["share_of_step"] = None
            extras["pgd"] = dict(public(m), metric="pgd_attacked_img_per_s", unit="img/s", scaling="weak", roofline=r_pgd,
                                 workload=WORKLOAD_TEXT["pgd"] % args.pgd_steps)
            log(f"[bench] pgd (batch {args.pgd_batch}/GPU): {m['value']:.1f} img/s")
            del dmp, m
        except Exception as ex:
            extras["pgd"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
        torch.cuda.empty_cache()
        if world == 1:
            ours = {"purify": main["value"]}
            for w2 in ("gender", "cars"):
                try:
                    t0 = time.perf_counter()
                    d2 = make_ours(w2, mode, dev)
                    m = measure(ctx, d2, w2, DEFAULT_BATCH[w2], 2, 3, mode, False)
                    extras[w2] = dict(public(m), metric="purified_img_per_s", unit="img/s", workload=WORKLOAD_TEXT[w2])
                    ours[w2] = m["value"]
                    log(f"[bench] {w2}: {m['value']:.1f} img/s ({time.perf_counter() - t0:.0f} s incl. model build)")
                    del d2, m
                except Exception as ex:
                    extras[w2] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
                torch.cuda.empty_cache()
            if not args.no_incumbent:
                t0 = time.perf_counter()
                extras["incumbent_gpu"] = incumbent_gpu(dev, ours=ours)
                log(f"[bench] incumbent_gpu: {time.perf_counter() - t0:.0f} s")
    elif args.incumbent and world == 1:
        extras["incumbent_gpu"] = incumbent_gpu(dev, workloads=("purify" if pgd else wl,), ours={("purify" if pgd else wl): main["value"]} if not pgd else None)

    if rank == 0:
        cpu = cpu_baseline() if not args.no_cpu_baseline else None
        line = {"metric": "pgd_attacked_img_per_s" if pgd else "purified_img_per_s", "value": main["value"], "unit": "img/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": mode, "data": "synthetic",
                "config": {"workload": (WORKLOAD_TEXT[wl] % args.pgd_steps) if pgd else WORKLOAD_TEXT[wl],
                           "nvae": None if sg else NVAE_C32_CONFIG, "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                           "l2": "no explicit flush: each step streams > 10 GB of activations through the 126 MB L2",
                           "cuda_graph": main["cuda_graph"], "streams": n_streams, "gflop_per_image_algorithmic": main["gflop_per_image_algorithmic"]},
                "tflops_algorithmic": main["tflops_algorithmic"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
                "hbm_peak_gb": main["hbm_peak_gb"], "clocks": main["clocks"], "roofline": roof, "roofline_other_kernels": extra,
                "cpu_baseline": cpu, "counters": main["counters"]}
        line.update(extras)
        print(json.dumps(line), file=JSON_OUT or sys.stdout, flush=True)
    if world > 1:
        ctx.dist.destroy_process_group()


JSON_OUT = None          # the process's original stdout; file descriptor 1 itself is pointed at stderr (see main)


def main():
    # stdout carries exactly ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its version banner
    # there even with NCCL_DEBUG_FILE set), so fd 1 is redirected to stderr for the whole run and the JSON goes to a dup of the original.
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--streams", type=int, default=0, help="part-batches / CUDA streams per call (0: 2 for purify and pgd, 1 otherwise)")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step (default 512 purify / 1024 pgd: 95 GB of tape + activations)")
    ap.add_argument("--workload", default="purify", choices=["purify", "pgd", "gender", "cars"])
    ap.add_argument("--chunk", type=int, default=0, help="generator batch chunk of the StyleGAN workloads (0: automatic)")
    ap.add_argument("--pgd-steps", type=int, default=50)
    ap.add_argument("--pgd-batch", type=int, default=256, help="images per GPU of the `pgd` extra block of the default line")
    ap.add_argument("--cuda-graph", type=int, default=-1, help="1: replay the call / PGD iteration as a CUDA graph; 0: eager; default: purify and pgd")
    ap.add_argument("--extras", type=int, default=1, help="default workload: also measure strong scaling, PGD, gender, cars and the incumbent-GPU bar")
    ap.add_argument("--incumbent", action="store_true", help="non-default workloads: add the incumbent-GPU block for this workload")
    ap.add_argument("--no-incumbent", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=0, help="bounded sample per step of the CPU reference arm (default 64 ids / 2 StyleGAN)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="CUDA-event time of EVERY op of the instrumented pass (table on stderr)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours: the reference arm draws fresh noise on every call")
        args.steps = args.steps if args.steps is not None else 4
        args.warmup = args.warmup if args.warmup is not None else 1
        run_reference(args)
    else:
        args.steps = args.steps if args.steps is not None else {"purify": 10, "pgd": 2}.get(args.workload, 3)
        args.warmup = args.warmup if args.warmup is not None else {"purify": 3, "pgd": 3}.get(args.workload, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
