"""CUDA-event timing of single ops at the attack-path / purify-path shapes (isolated, L2-flushed between launches):
python scripts/bench_ops.py [dwconv] [mbconv] [k1] [hbm] [level]"""
import sys
import torch
sys.path.insert(0, ".")
from gen_adversarial_b200 import ops
from gen_adversarial_b200._lib import ACT_NONE, ACT_SILU

DEV = "cuda:0"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def dwconv():
    g = torch.Generator(device=DEV).manual_seed(0)
    for (n, h, c, up) in [(128, 32, 384, False), (128, 16, 768, False), (128, 8, 1536, False), (512, 64, 96, False),
                          (512, 16, 768, True), (512, 32, 192, True), (512, 8, 1536, True)]:
        x = torch.randn(n, h, h, c, device=DEV, generator=g).bfloat16()
        w = torch.randn(25, c, device=DEV, generator=g) * 0.2
        b = torch.randn(c, device=DEV, generator=g) * 0.1
        s = 2 if up else 1
        m = torch.randn(n, h * s, h * s, c, device=DEV, generator=g).bfloat16()
        elems_out = n * h * s * h * s * c
        elems_in = n * h * h * c
        t_plain = timeit(lambda: ops.dwconv5x5(x, w, b, ACT_SILU, up, torch.bfloat16))
        t_tape = timeit(lambda: ops.dwconv5x5(x, w, b, ACT_SILU, up, torch.bfloat16, want_dact=True))
        t_bwd = timeit(lambda: ops.dwconv5x5(x, w, None, ACT_NONE, up, torch.bfloat16, mul=m)) if not up else float("nan")
        gb = lambda k_out, t: (elems_in * 2 + k_out * elems_out * 2) / t / 1e3
        print(f"dwconv n={n} hw={h} c={c} up={int(up)}: plain {t_plain:7.1f} us ({gb(1, t_plain):5.0f} GB/s)  taping {t_tape:7.1f} us "
              f"({gb(2, t_tape):5.0f} GB/s)  backward {t_bwd:7.1f} us ({gb(2, t_bwd):5.0f} GB/s)   FMA floor {elems_out * 25 / (148 * 128 * 1.965e3):6.1f} us")


def mbconv():
    import math
    g = torch.Generator(device=DEV).manual_seed(0)
    for (n, w, c) in [(512, 32, 64), (512, 16, 128), (512, 8, 256)]:
        hidden = 6 * c
        e = ops.ConvLayer(1, 1, 1, 0, c, hidden, post_act=ACT_SILU, name="expand")
        e.w_tc = (torch.randn(hidden, c, device=DEV, generator=g) / math.sqrt(c)).bfloat16().contiguous()
        e.bias = torch.randn(hidden, device=DEV, generator=g) * 0.3
        p = ops.ConvLayer(1, 1, 1, 0, hidden, c, post_act=ACT_NONE, name="project")
        p.w_tc = (torch.randn(c, hidden, device=DEV, generator=g) / math.sqrt(hidden)).bfloat16().contiguous()
        p.bias = torch.randn(c, device=DEV, generator=g) * 0.3
        dw = ops.dw_weights_chunked(torch.randn(25, hidden, device=DEV, generator=g) / 5.0)
        db = torch.randn(hidden, device=DEV, generator=g) * 0.3
        x = torch.randn(n, w, w, c, device=DEV, generator=g).bfloat16()
        t = timeit(lambda: ops.mbconv_fused(x, e, dw, db, p))
        m = n * w * w
        fl = 2.0 * m * hidden * c * 2 + 2.0 * m * hidden * 25
        print(f"mbconv n={n} hw={w} c={c} hidden={hidden}: {t:7.1f} us  {fl / t / 1e6:6.1f} TFLOP/s   fp32-pipe floor "
              f"{m * hidden * (25 + 5) / (148 * 128 * 1.965e3):6.1f} us")
        # attack path: taping forward and backward of the cell, fused against the three kernels each replaces
        t_tape = timeit(lambda: ops.mbconv_fused(x, e, dw, db, p, want_sums=True, want_tape=True))
        dw_w = dw.permute(1, 0, 2).reshape(25, hidden).contiguous()

        def tape3():
            de = torch.empty(n, w, w, hidden, device=DEV, dtype=torch.bfloat16)
            h1, _ = ops.conv2d_tc(x, e, dact_out=de)
            h2, dd = ops.dwconv5x5(h1, dw_w, db, ACT_SILU, False, torch.bfloat16, want_dact=True)
            r, _ = ops.conv2d_tc(h2, p)
            return ops.channel_sum(r)
        t_tape3 = timeit(tape3)
        _, _, de, dd = ops.mbconv_fused(x, e, dw, db, p, want_sums=True, want_tape=True)
        p_d = ops.ConvLayer(1, 1, 1, 0, c, hidden, post_act=ACT_NONE, name="project_dgrad")
        p_d.w_tc = p.w_tc.t().contiguous()
        e_d = ops.ConvLayer(1, 1, 1, 0, hidden, c, post_act=ACT_NONE, name="expand_dgrad")
        e_d.w_tc = e.w_tc.t().contiguous()
        dw_wT = dw_w.flip(0).contiguous()
        dwTc = ops.dw_weights_chunked(dw_wT)
        gr = (torch.randn(n, w, w, c, device=DEV, generator=g) * 1e-3).bfloat16()
        add = torch.randn(n, w, w, c, device=DEV, generator=g) * 1e-3
        t_bwd = timeit(lambda: ops.mbconv_fused_bwd(gr, p_d, dwTc, dd, de, e_d, add=add))

        def bwd3():
            g2, _ = ops.conv2d_tc(gr, p_d, mul=dd)
            g1 = ops.dwconv5x5(g2, dw_wT, None, ACT_NONE, False, torch.bfloat16, mul=de)
            return ops.conv2d_tc(g1, e_d, want_bf16=False, want_f32=True, add=add)
        t_bwd3 = timeit(bwd3)
        print(f"   attack path: taping fwd fused {t_tape:7.1f} us (three kernels + channel_sum {t_tape3:7.1f} us)   backward fused {t_bwd:7.1f} us "
              f"(three kernels {t_bwd3:7.1f} us)")
        del de, dd


def k1():
    """the 1x1 convs of the attack path's decoder cells: expand with SiLU + saved derivative, dgrad of the project conv times a saved
    derivative, project; plus the 3x3 tower conv for reference"""
    import math
    g = torch.Generator(device=DEV).manual_seed(0)
    for (n, w, c) in [(512, 32, 64), (512, 16, 128), (512, 8, 256)]:
        hidden = 6 * c
        m = n * w * w
        x = torch.randn(n, w, w, c, device=DEV, generator=g).bfloat16()
        hbig = torch.randn(n, w, w, hidden, device=DEV, generator=g).bfloat16()
        e = ops.ConvLayer(1, 1, 1, 0, c, hidden, post_act=ACT_SILU, name="expand")
        e.w_tc = (torch.randn(hidden, c, device=DEV, generator=g) / math.sqrt(c)).bfloat16().contiguous()
        e.bias = torch.randn(hidden, device=DEV, generator=g) * 0.3
        pd = ops.ConvLayer(1, 1, 1, 0, c, hidden, post_act=ACT_NONE, name="project.dgrad")
        pd.w_tc = e.w_tc
        pr = ops.ConvLayer(1, 1, 1, 0, hidden, c, post_act=ACT_NONE, name="project")
        pr.w_tc = (torch.randn(c, hidden, device=DEV, generator=g) / math.sqrt(hidden)).bfloat16().contiguous()
        pr.bias = torch.randn(c, device=DEV, generator=g) * 0.3
        k3 = ops.ConvLayer(3, 3, 1, 1, c, c, post_act=ACT_SILU, name="k3")
        k3.w_tc = (torch.randn(c, 9 * c, device=DEV, generator=g) / math.sqrt(9 * c)).bfloat16().contiguous()
        k3.bias = torch.randn(c, device=DEV, generator=g) * 0.3
        dact = torch.empty(n, w, w, hidden, device=DEV, dtype=torch.bfloat16)
        ob = torch.empty(n, w, w, hidden, device=DEV, dtype=torch.bfloat16)
        os_ = torch.empty(n, w, w, c, device=DEV, dtype=torch.bfloat16)
        t_plain = timeit(lambda: ops.conv2d_tc(x, e, out_bf16=ob))
        t_tape = timeit(lambda: ops.conv2d_tc(x, e, dact_out=dact, out_bf16=ob))
        t_dg = timeit(lambda: ops.conv2d_tc(x, pd, mul=hbig, out_bf16=ob))
        t_pr = timeit(lambda: ops.conv2d_tc(hbig, pr, out_bf16=os_))
        t_k3 = timeit(lambda: ops.conv2d_tc(x, k3, out_bf16=os_))
        big, small = m * hidden * 2, m * c * 2
        print(f"k1 n={n} hw={w} c={c}: expand {t_plain:6.1f} us ({(small + big) / t_plain / 1e3:5.0f} GB/s)  expand+dact {t_tape:6.1f} us "
              f"({(small + 2 * big) / t_tape / 1e3:5.0f} GB/s)  dgrad*mul {t_dg:6.1f} us ({(small + 2 * big) / t_dg / 1e3:5.0f} GB/s)  "
              f"project {t_pr:6.1f} us ({(small + big) / t_pr / 1e3:5.0f} GB/s)  k3 {t_k3:6.1f} us ({2.0 * m * c * 9 * c / t_k3 / 1e6:5.0f} TFLOP/s)")


def hbm():
    """the HBM-bound fused elementwise / stencil kernels (north-star item 3) at the BASELINE batch and at a saturating batch:
    achieved GB/s on the ALGORITHMIC bytes of SURVEY 8d against the measured copy peak"""
    import json, os
    peak = 6542.1
    try:
        peak = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    g = torch.Generator(device=DEV).manual_seed(0)

    def report(name, us, nbytes):
        gbs = nbytes / us / 1e3
        print(f"{name:58s} {us:8.1f} us  {nbytes / 1e6:8.1f} MB  {gbs:7.0f} GB/s  {100 * gbs / peak:5.1f}% of {peak:.0f}")

    for n in (512, 4096):
        x = torch.rand(n, 3, 64, 64, device=DEV, generator=g)
        by = 2 * x.numel() * 4
        report(f"preprocess blur (R=7) batch {n}", timeit(lambda: ops.preprocess(x, None, 0.0, True, torch.bfloat16)), x.numel() * 4 + x.numel() * 2)
        report(f"preprocess Philox noise batch {n}", timeit(lambda: ops.preprocess(x, None, 1.0, False, torch.bfloat16, seed=3)), x.numel() * 4 + x.numel() * 2)
        adv, gr = x.clone(), torch.randn(x.shape, device=DEV, generator=g)
        report(f"pgd_linf_step batch {n}", timeit(lambda: ops.pgd_linf_step_(adv, gr, x, 2 / 255, 8 / 255)), 4 * x.numel() * 4)
        del adv, gr
    alpha = torch.tensor([0.5], device=DEV)
    for n in (512, 2048):
        for hw in (32, 16, 8):
            q = torch.randn(n, hw, hw, 24, device=DEV, generator=g)
            pp = torch.randn(n, hw, hw, 40, device=DEV, generator=g)
            t = timeit(lambda: ops.latent_mix(q, pp, None, 5, 3, 0, alpha, 0.6, 20, 24, torch.bfloat16))
            report(f"latent_mix (Philox eps) n={n} hw={hw}", t, n * hw * hw * (20 * 4 + 40 * 4 + 20 * 2))
        logits = torch.randn(n, 64, 64, 100, device=DEV, generator=g)
        t = timeit(lambda: ops.discmix_mean(logits, 10, torch.bfloat16))
        report(f"discmix_mean n={n} (100 fp32 logits -> NCHW fp32 + NHWC bf16)", t, n * 4096 * (100 * 4 + 3 * 4 + 3 * 2))
        del logits
    for (n, hw, c) in [(512, 32, 64), (512, 16, 128), (512, 8, 256), (2048, 32, 64)]:
        r = torch.randn(n, hw, hw, c, device=DEV, generator=g).bfloat16()
        skip = torch.randn(n, hw, hw, c, device=DEV, generator=g)
        hid = max(c // 16, 4)
        se = (torch.randn(hid, c, device=DEV, generator=g) * 0.3, torch.randn(hid, device=DEV, generator=g) * 0.1,
              torch.randn(c, hid, device=DEV, generator=g) * 0.3, torch.randn(c, device=DEV, generator=g) * 0.1)
        sums = ops.channel_sum(r)
        e = r.numel()
        report(f"channel_sum n={n} hw={hw} c={c}", timeit(lambda: ops.channel_sum(r)), e * 2)
        report(f"se_residual (fp32 stream + bf16 copy) n={n} hw={hw} c={c}",
               timeit(lambda: ops.se_residual(r, sums, se, 0.1, skip, torch.float32, want_out2=True)), e * (2 + 4 + 4 + 2))
        go = torch.randn(n, hw, hw, c, device=DEV, generator=g)
        report(f"se_residual_bwd n={n} hw={hw} c={c}", timeit(lambda: ops.se_residual_bwd(go, r, sums, se, 0.1, torch.bfloat16)), e * (2 * (4 + 2) + 2))
        del r, skip, go


def level():
    """tail of one decoder latent level at batch 512, per level size: the three launches (sampler 1x1 -> latent_mix -> combiner 1x1 with z as
    second source) against the fused latent_level kernel.  GB/s on the fused pass's compulsory bytes (x_elu and xa bf16, muq fp32 in; the
    stream fp32 + bf16 out), against a device-to-device copy timed in the same process."""
    import math
    g = torch.Generator(device=DEV).manual_seed(0)
    src = torch.empty(1 << 30, dtype=torch.uint8, device=DEV)
    dst = torch.empty_like(src)
    peak = 2 * src.numel() / timeit(lambda: dst.copy_(src)) / 1e3
    del src, dst
    print(f"device-to-device copy: {peak:.0f} GB/s (read + write)")
    zdim, zc, temp = 20, 24, 0.6
    alpha = torch.full((1,), 0.5, device=DEV)
    for (n, hw, c) in [(512, 32, 64), (512, 16, 128), (512, 8, 256)]:
        smp = ops.ConvLayer(1, 1, 1, 0, c, 2 * zdim, name="dec_sampler")
        smp.w_tc = (torch.randn(2 * zdim, c, device=DEV, generator=g) * (0.7 / math.sqrt(c))).bfloat16().contiguous()
        smp.bias = torch.randn(2 * zdim, device=DEV, generator=g) * 0.2
        comb = ops.ConvLayer(1, 1, 1, 0, c, c, cin2=zc, name="dec_comb")
        comb.w_tc = (torch.randn(c, c + zc, device=DEV, generator=g) / math.sqrt(c + zdim)).bfloat16().contiguous()
        comb.bias = torch.randn(c, device=DEV, generator=g) * 0.2
        x_elu = torch.nn.functional.elu(torch.randn(n, hw, hw, c, device=DEV, generator=g)).bfloat16()
        xa = torch.randn(n, hw, hw, c, device=DEV, generator=g).bfloat16()
        muq = torch.randn(n, hw, hw, zdim, device=DEV, generator=g)

        def three():
            pp = ops.conv2d_tc(x_elu, smp, want_bf16=False, want_f32=True)[1]
            z = ops.latent_mix(muq, pp, None, 5, 3, 0, alpha, temp, zdim, zc, torch.bfloat16)
            return ops.conv2d_tc(xa, comb, want_bf16=True, want_f32=True, x2=z)

        t3 = timeit(three)
        t1 = timeit(lambda: ops.latent_level(x_elu, xa, muq, None, smp, comb, 5, 3, 0, alpha, temp, zdim))
        t1p = timeit(lambda: ops.latent_level(x_elu, xa, muq, None, smp, comb, 5, 3, 0, alpha, temp, zdim, want_pp=True))
        m = n * hw * hw
        by = m * (2 * c + 2 * c + 4 * zdim + 6 * c)
        gbs = by / t1 / 1e3
        print(f"level n={n} hw={hw} c={c}: three launches {t3:7.1f} us  fused {t1:7.1f} us ({by / 1e6:6.1f} MB, {gbs:5.0f} GB/s, "
              f"{100 * gbs / peak:4.1f}% of copy)  fused + pp tape {t1p:7.1f} us  speed-up {t3 / t1:4.2f}x")


if __name__ == "__main__":
    which = sys.argv[1:] or ["dwconv"]
    if "dwconv" in which:
        dwconv()
    if "mbconv" in which:
        mbconv()
    if "k1" in which:
        k1()
    if "hbm" in which:
        hbm()
    if "level" in which:
        level()
