"""TEST INFRASTRUCTURE ONLY -- CPU restatement (plain torch ops on the reference's own, unfolded `state_dict`s) of the
StyleGAN purification paths: BASELINE configs 3 (E4E @1024 + ResNet-50) and 4 (Style-Transformer @512 + ResNeXt-50).

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may import this module.
Pinned against the UNMODIFIED reference by tests/test_oracle_vs_reference.py (shimmed import, oracle/ref_import.py) and by
the fixtures tests/golden/e4e_gender_b1.pt / trans_cars_b1.pt that oracle/make_golden.py produced from the reference.
Paths cited are relative to /root/reference/src/.  kornia / torchvision arithmetic is third-party and unpinned
(environment.yml:17): restated semantics are listed in oracle/ref_import.py; ResNet bodies follow torchvision 0.26.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

BN_EPS = 1e-5
IRSE50_BLOCKS = [(64, 64, 3), (64, 128, 4), (128, 256, 14), (256, 512, 3)]     # mlvgms_autoencoders/StyleGan_E4E/encoding/helpers.py:30-37


def _bn(sd, p, x):
    return F.batch_norm(x, sd[f"{p}.running_mean"], sd[f"{p}.running_var"], sd[f"{p}.weight"], sd[f"{p}.bias"], False, 0.0, BN_EPS)


def _sub(sd, prefix):
    n = len(prefix) + 1
    return {k[n:]: v for k, v in sd.items() if k.startswith(prefix + ".")}       # get_keys, StyleGan_E4E/psp.py:8-12


# ------------------------------------------------------------------------------------------------ preprocessing (abstract_models.py:129-159)
def gaussian_blur(x):
    """defenses/ours/abstract_models.py:145-159 + kornia gaussian_blur2d (reflect border, separable, sigma 1)"""
    b, c, h, w = x.shape
    k = int(2 ** (math.sqrt(h) // 2) - 1)
    t = torch.arange(k, dtype=x.dtype) - k // 2
    g = torch.exp(-(t ** 2) / 2.0)
    g = g / g.sum()
    xp = F.pad(x, (k // 2, k // 2, k // 2, k // 2), mode="reflect")
    xp = F.conv2d(xp, g.view(1, 1, 1, k).expand(c, 1, 1, k), groups=c)
    return F.conv2d(xp, g.view(1, 1, k, 1).expand(c, 1, k, 1), groups=c)


def add_noise(x, noise, eps):
    """abstract_models.py:129-143 with the N(0,1) draw supplied explicitly"""
    nn_ = noise.flatten(1).norm(dim=1).view(-1, 1, 1, 1)
    return (x + noise * (eps / nn_)).clamp(0.0, 1.0)


# ------------------------------------------------------------------------------------------------ IR-SE50 (encoding/helpers.py:57-120)
def irse50_backbone(sd: Dict[str, torch.Tensor], x: torch.Tensor):
    """`input_layer` + 24 `bottleneck_IR_SE`; taps after units 6, 20, 23 (encoding/encoder.py:110-124)"""
    x = F.prelu(_bn(sd, "input_layer.1", F.conv2d(x, sd["input_layer.0.weight"], padding=1)), sd["input_layer.2.weight"])
    taps = {}
    i = 0
    for cin0, depth, n in IRSE50_BLOCKS:
        for j in range(n):
            stride = 2 if j == 0 else 1
            p = f"body.{i}"
            if f"{p}.shortcut_layer.0.weight" in sd:
                sc = _bn(sd, f"{p}.shortcut_layer.1", F.conv2d(x, sd[f"{p}.shortcut_layer.0.weight"], stride=stride))
            else:
                sc = x[:, :, ::stride, ::stride]                                         # MaxPool2d(1, stride)
            r = _bn(sd, f"{p}.res_layer.0", x)
            r = F.prelu(F.conv2d(r, sd[f"{p}.res_layer.1.weight"], padding=1), sd[f"{p}.res_layer.2.weight"])
            r = _bn(sd, f"{p}.res_layer.4", F.conv2d(r, sd[f"{p}.res_layer.3.weight"], stride=stride, padding=1))
            s = r.mean(dim=(2, 3), keepdim=True)                                         # SEModule, helpers.py:57-74
            s = torch.sigmoid(F.conv2d(F.relu(F.conv2d(s, sd[f"{p}.res_layer.5.fc1.weight"])), sd[f"{p}.res_layer.5.fc2.weight"]))
            x = r * s + sc
            if i in (6, 20, 23):
                taps[i] = x
            i += 1
    return taps[6], taps[20], taps[23]


def _upsample_add(x, y):
    return F.interpolate(x, size=y.shape[-2:], mode="bilinear", align_corners=True) + y   # helpers.py:122-139


def e4e_encode(sd, x, stylegan_size: int, latent_avg: Optional[torch.Tensor]):
    """`Encoder4Editing.forward` at Inference stage (encoder.py:110-140) + `pSp.encode` (psp.py:88-101)"""
    c1, c2, c3 = irse50_backbone(sd, x)
    n_styles = 2 * int(math.log2(stylegan_size)) - 2

    def head(i, feat):                                                                   # GradualStyleBlock, encoder.py:33-54
        spatial = 16 if i < 3 else (32 if i < 7 else 64)
        h = feat
        for j in range(int(math.log2(spatial))):
            h = F.leaky_relu(F.conv2d(h, sd[f"styles.{i}.convs.{2 * j}.weight"], sd[f"styles.{i}.convs.{2 * j}.bias"], stride=2, padding=1), 0.01)
        h = h.reshape(-1, 512)
        return F.linear(h, sd[f"styles.{i}.linear.weight"] * (1.0 / math.sqrt(512)), sd[f"styles.{i}.linear.bias"])

    w0 = head(0, c3)
    w = w0.unsqueeze(1).repeat(1, n_styles, 1)
    feat = c3
    for i in range(1, n_styles):
        if i == 3:
            p2 = _upsample_add(c3, F.conv2d(c2, sd["latlayer1.weight"], sd["latlayer1.bias"]))
            feat = p2
        elif i == 7:
            feat = _upsample_add(p2, F.conv2d(c1, sd["latlayer2.weight"], sd["latlayer2.bias"]))
        w[:, i] = w[:, i] + head(i, feat)
    if latent_avg is not None:
        w = w + latent_avg.unsqueeze(0)
    return w


# ------------------------------------------------------------------------------------------------ Style-Transformer encoder
def _mha(sd, p, q_in, k_in, v_in, heads=4):
    """torch.nn.MultiheadAttention forward (eval, no masks); tensors (L, B, E)"""
    e = q_in.shape[-1]
    w, b = sd[f"{p}.in_proj_weight"], sd[f"{p}.in_proj_bias"]
    q = F.linear(q_in, w[:e], b[:e])
    k = F.linear(k_in, w[e:2 * e], b[e:2 * e])
    v = F.linear(v_in, w[2 * e:], b[2 * e:])
    lq, bsz, _ = q.shape
    dh = e // heads
    q = q.reshape(lq, bsz * heads, dh).transpose(0, 1) / math.sqrt(dh)
    k = k.reshape(-1, bsz * heads, dh).transpose(0, 1)
    v = v.reshape(-1, bsz * heads, dh).transpose(0, 1)
    a = torch.softmax(q @ k.transpose(1, 2), dim=-1) @ v
    a = a.transpose(0, 1).reshape(lq, bsz, e)
    return F.linear(a, sd[f"{p}.out_proj.weight"], sd[f"{p}.out_proj.bias"])


def transformer_decoder_layer(sd, p, tgt, memory):
    """`TransformerDecoderLayer.forward_post` (StyleGan_Trans/models/transformer.py:40-66), dropout inactive in eval"""
    ln = lambda k, t: F.layer_norm(t, (t.shape[-1],), sd[f"{p}.norm{k}.weight"], sd[f"{p}.norm{k}.bias"], 1e-5)
    tgt = ln(1, tgt + _mha(sd, f"{p}.self_attn", tgt, tgt, tgt))
    tgt = ln(2, tgt + _mha(sd, f"{p}.multihead_attn", tgt, memory, memory))
    ff = F.linear(F.relu(F.linear(tgt, sd[f"{p}.linear1.weight"], sd[f"{p}.linear1.bias"])), sd[f"{p}.linear2.weight"], sd[f"{p}.linear2.bias"])
    return ln(3, tgt + ff)


def trans_encode(sd, x, query, latent_avg):
    """`GradualStyleEncoder.forward` (encoders/style_transformer_encoders.py:61-84) + latent_avg (defenses/ours/models.py:318-325)"""
    c1, c2, c3 = irse50_backbone(sd, x)
    p2 = _upsample_add(c3, F.conv2d(c2, sd["latlayer1.weight"], sd["latlayer1.bias"]))
    p1 = _upsample_add(p2, F.conv2d(c1, sd["latlayer2.weight"], sd["latlayer2.bias"]))
    tok = lambda t: t.flatten(2).permute(2, 0, 1)
    q = query.permute(1, 0, 2)
    q = transformer_decoder_layer(sd, "transformerlayer_coarse", q, tok(c3))
    q = transformer_decoder_layer(sd, "transformerlayer_medium", q, tok(p2))
    q = transformer_decoder_layer(sd, "transformerlayer_fine", q, tok(p1))
    codes = q.permute(1, 0, 2)
    if latent_avg is not None:
        codes = codes + latent_avg.unsqueeze(0)
    return codes


# ------------------------------------------------------------------------------------------------ StyleGAN2 generator
def fused_leaky_relu(x, bias):
    """stylegan2/op/fused_bias_act_kernel.cu:28-47"""
    if bias is not None:
        x = x + bias.view(1, -1, *([1] * (x.dim() - 2)))
    return F.leaky_relu(x, 0.2) * math.sqrt(2.0)


def upfirdn2d(x, kernel, up=1, down=1, pad=(0, 0)):
    """stylegan2/op/upfirdn2d_kernel.cu:52-137 (zero-insert, pad, correlate with the flipped FIR, decimate)"""
    b, c, h, w = x.shape
    kh, kw = kernel.shape
    y = x.reshape(b * c, 1, h, 1, w, 1)
    y = F.pad(y, [0, up - 1, 0, 0, 0, up - 1]).reshape(b * c, 1, h * up, w * up)
    y = F.pad(y, [pad[0], pad[1], pad[0], pad[1]])
    y = F.conv2d(y, torch.flip(kernel, [0, 1]).view(1, 1, kh, kw).to(y.dtype))
    y = y[:, :, ::down, ::down]
    return y.reshape(b, c, y.shape[2], y.shape[3])


def generator_style(sd, z, n_mlp=8, lr_mlp=0.01):
    """`Generator.style`: PixelNorm + 8 x EqualLinear(fused_lrelu) (stylegan2/generator.py:10-15,69-100,311-320)"""
    x = z * torch.rsqrt(torch.mean(z ** 2, dim=1, keepdim=True) + 1e-8)
    d = z.shape[1]
    for i in range(1, n_mlp + 1):
        x = F.linear(x, sd[f"style.{i}.weight"] * ((1.0 / math.sqrt(d)) * lr_mlp))
        x = fused_leaky_relu(x, sd[f"style.{i}.bias"] * lr_mlp)
    return x


def _modconv(sd, p, x, style, demodulate, upsample):
    """`ModulatedConv2d.forward` (stylegan2/generator.py:163-207): per-sample weights, grouped conv with groups = batch"""
    w = sd[f"{p}.weight"]                                                              # (1, cout, cin, k, k)
    _, cout, cin, k, _ = w.shape
    b, _, h, wd = x.shape
    s = F.linear(style, sd[f"{p}.modulation.weight"] * (1.0 / math.sqrt(style.shape[1])), sd[f"{p}.modulation.bias"])
    weight = (1.0 / math.sqrt(cin * k * k)) * w * s.view(b, 1, cin, 1, 1)
    if demodulate:
        weight = weight * torch.rsqrt(weight.pow(2).sum([2, 3, 4]) + 1e-8).view(b, cout, 1, 1, 1)
    if upsample:
        wt = weight.transpose(1, 2).reshape(b * cin, cout, k, k)
        out = F.conv_transpose2d(x.reshape(1, b * cin, h, wd), wt, padding=0, stride=2, groups=b)
        out = out.view(b, cout, out.shape[2], out.shape[3])
        return upfirdn2d(out, sd[f"{p}.blur.kernel"], pad=(1, 1))                       # pad0 = pad1 = 1 for k = 3, generator.py:131-136
    out = F.conv2d(x.reshape(1, b * cin, h, wd), weight.view(b * cout, cin, k, k), padding=k // 2, groups=b)
    return out.view(b, cout, out.shape[2], out.shape[3])


def generator_synthesis(sd, latent, size: int):
    """`Generator.forward(input_is_latent=True, randomize_noise=False)` (stylegan2/generator.py:407-479)"""
    log_size = int(math.log2(size))

    def styled(p, x, st, noise, up):
        out = _modconv(sd, f"{p}.conv", x, st, True, up)
        out = out + sd[f"{p}.noise.weight"] * noise
        return fused_leaky_relu(out, sd[f"{p}.activate.bias"])

    def to_rgb(p, x, st, skip):
        out = _modconv(sd, f"{p}.conv", x, st, False, False) + sd[f"{p}.bias"]
        if skip is not None:
            out = out + upfirdn2d(skip, sd[f"{p}.upsample.kernel"], up=2, pad=(2, 1))   # Upsample, generator.py:28-47
        return out

    b = latent.shape[0]
    x = sd["input.input"].repeat(b, 1, 1, 1)
    x = styled("conv1", x, latent[:, 0], sd["noises.noise_0"], False)
    skip = to_rgb("to_rgb1", x, latent[:, 1], None)
    i = 1
    for j in range(log_size - 2):
        x = styled(f"convs.{2 * j}", x, latent[:, i], sd[f"noises.noise_{2 * j + 1}"], True)
        x = styled(f"convs.{2 * j + 1}", x, latent[:, i + 1], sd[f"noises.noise_{2 * j + 2}"], False)
        skip = to_rgb(f"to_rgbs.{j}", x, latent[:, i + 2], skip)
        i += 2
    return skip


def mix_codes(sd_dec, codes, z_noise, alphas):
    """per-level latent interpolation, defenses/ours/models.py:117-127 / 329-342; z_noise (n, B, d) already scaled by its std"""
    styles = torch.stack([generator_style(sd_dec, n) for n in z_noise], dim=0)
    a = torch.tensor(alphas, dtype=codes.dtype, device=codes.device).view(-1, 1, 1)
    return ((1 - a) * codes.permute(1, 0, 2) + a * styles).permute(1, 0, 2)


# ------------------------------------------------------------------------------------------------ classifiers
def resnet_forward(sd, x, groups: int = 1):
    """`ResNet` / `ResNext` (classifier/model.py:10-28,53-70): torchvision resnet50 / resnext50_32x4d + 4-layer head, eval mode"""
    sd = {(k[len("model."):] if k.startswith("model.") else k): v for k, v in sd.items()}
    x = F.relu(_bn(sd, "bn1", F.conv2d(x, sd["conv1.weight"], stride=2, padding=3)))
    x = F.max_pool2d(x, 3, 2, 1)
    for li, n in enumerate((3, 4, 6, 3), start=1):
        for bi in range(n):
            p = f"layer{li}.{bi}"
            stride = 2 if (li > 1 and bi == 0) else 1
            h = F.relu(_bn(sd, f"{p}.bn1", F.conv2d(x, sd[f"{p}.conv1.weight"])))
            h = F.relu(_bn(sd, f"{p}.bn2", F.conv2d(h, sd[f"{p}.conv2.weight"], stride=stride, padding=1, groups=groups)))
            h = _bn(sd, f"{p}.bn3", F.conv2d(h, sd[f"{p}.conv3.weight"]))
            idt = x
            if f"{p}.downsample.0.weight" in sd:
                idt = _bn(sd, f"{p}.downsample.1", F.conv2d(x, sd[f"{p}.downsample.0.weight"], stride=stride))
            x = F.relu(h + idt)
    x = x.mean(dim=(2, 3))
    x = F.relu(_bn(sd, "fc.1", F.linear(x, sd["fc.0.weight"])))
    return F.linear(x, sd["fc.3.weight"], sd["fc.3.bias"])


# ------------------------------------------------------------------------------------------------ whole defense calls (abstract_models.py:161-193)
def _preprocess(x, noise0, eps, blur):
    if blur:
        x = gaussian_blur(x)
    x = add_noise(x, noise0, eps)                       # the reference draws and adds noise even when eps = 0
    return (x - 0.5) / 0.5


def e4e_defense_call(ckpt, clf_sd, x, alphas, noises: List[torch.Tensor], eps: float, blur: bool):
    """`E4EStyleGanDefenseModel.__call__` (models.py:79-132): x (B,3,256,256) in [0,1]; noises = [N(0,1) (B,3,256,256), N(0,1) (18,B,512)]
    -> (logits, purified in [0,1])"""
    sd = ckpt["state_dict"]
    enc, dec = _sub(sd, "encoder"), _sub(sd, "decoder")
    size = ckpt["opts"]["stylegan_size"]
    xn = _preprocess(x, noises[0], eps, blur)
    codes = e4e_encode(enc, xn, size, ckpt.get("latent_avg"))
    codes = mix_codes(dec, codes, noises[1], alphas)
    img = generator_synthesis(dec, codes, size)
    img = F.adaptive_avg_pool2d(img, (256, 256))                                       # face_pool, psp.py:26,114
    purified = img * 0.5 + 0.5
    logits = resnet_forward(clf_sd, (purified - 0.5) / 0.5, 1) if clf_sd is not None else None
    return logits, purified


def trans_defense_call(ckpt, clf_sd, x, alphas, noises: List[torch.Tensor], eps: float, blur: bool):
    """`TransStyleGanDefenseModel.__call__` (models.py:277-353): x (B,3,128,128) in [0,1]; noises = [N(0,1) (B,3,128,128), N(0,1) (16,B,512)]"""
    sd = ckpt["state_dict"]
    enc, dec = _sub(sd, "encoder.module"), _sub(sd, "decoder.module")
    size = ckpt["opts"]["output_size"]
    xn = _preprocess(x, noises[0], eps, blur)
    xr = F.interpolate(xn, size=(256, 256), mode="bilinear", align_corners=False)[:, :, 32:-32]    # kornia resize + crop, models.py:307-308
    z = enc["z"]
    b = x.shape[0]
    query = generator_style(dec, z.expand(b, -1, -1).flatten(0, 1)).reshape(b, z.shape[1], z.shape[2])
    codes = trans_encode(enc, xr, query, ckpt.get("latent_avg"))
    codes = mix_codes(dec, codes, noises[1] * 0.8, alphas)                             # torch.normal(0, 0.8, ...), models.py:334
    img = generator_synthesis(dec, codes, size)
    img = F.adaptive_avg_pool2d(img, (256, 256))
    img[:, :, :32] = -1.0
    img[:, :, -32:] = -1.0
    img = F.interpolate(img, size=(128, 128), mode="bilinear", align_corners=False)    # kornia resize(images, 128), models.py:351
    purified = img * 0.5 + 0.5
    logits = resnet_forward(clf_sd, (purified - 0.5) / 0.5, 32) if clf_sd is not None else None
    return logits, purified
