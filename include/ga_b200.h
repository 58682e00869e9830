/*
 * ga_b200.h -- C ABI of libga_b200.so: hand-written sm_100a CUDA kernels for the purification hot
 * path of SerezD/gen_adversarial (preprocess -> NVAE encode -> per-level latent mix -> decode ->
 * classify, plus the input-gradient backward and the fused PGD step).
 *
 * Conventions (SURVEY.md section 8b, last row):
 *   - extern "C", plain pointers and sizes; no C++/torch types cross the boundary.
 *   - The CALLER owns every buffer (PyTorch allocates, passes data_ptr()).  The library owns nothing
 *     between calls: every entry point is stateless, launches on the caller-supplied stream, never
 *     synchronises, and is CUDA-graph capturable.
 *   - Activations are dense NHWC (channels innermost).  The reference-facing boundary tensors
 *     (input batch, noise draws, purified images, gradients w.r.t. the batch) are NCHW fp32 exactly as
 *     the reference passes them (src/defenses/ours/abstract_models.py:161-193).
 *   - Return value 0 = ok; non-zero = error, message via ga_last_error() (thread-local).  The Python
 *     host raises RuntimeError -- mirrors TORCH_CHECK in the reference's
 *     src/mlvgms_autoencoders/StyleGan_E4E/stylegan2/op/fused_bias_act.cpp:7-9.
 *
 * Each entry point cites the reference code it replaces (paths relative to /root/reference).
 */
#ifndef GA_B200_H
#define GA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GA_ABI_VERSION 11

enum ga_dtype { GA_F32 = 0, GA_BF16 = 1 };
enum ga_pre_op { GA_PRE_NONE = 0, GA_PRE_ELU = 1, GA_PRE_SILU = 2, GA_PRE_AFFINE_SILU = 3, GA_PRE_AFFINE = 4 };
enum ga_act { GA_ACT_NONE = 0, GA_ACT_SILU = 1, GA_ACT_ELU = 2, GA_ACT_RELU = 3,
              GA_ACT_LRELU_SQRT2 = 4 /* leaky_relu(x, 0.2) * sqrt(2): fused_bias_act_kernel.cu:28-47 */,
              GA_ACT_PRELU = 5 /* x > 0 ? x : act_slope[c] * x (nn.PReLU / nn.LeakyReLU of the IR-SE50 encoder) */ };
/* epilogue multiplier modes (backward): multiply by the tensor itself, or by the ReLU / ELU derivative
 * reconstructed from the saved OUTPUT y of the forward activation (relu: y>0, elu: y>0 ? 1 : y+1) */
enum ga_mul_mode { GA_MUL_VALUE = 0, GA_MUL_RELU_MASK = 1, GA_MUL_ELU_FROM_Y = 2 };

/* dense NHWC tensor view */
typedef struct ga_tensor {
  void* data;
  int32_t dtype;          /* ga_dtype */
  int32_t n, h, w, c;
} ga_tensor;

/* convolution as implicit GEMM; weights already folded (weight-norm, eval-BN) by the host */
typedef struct ga_conv_desc {
  int32_t kh, kw;         /* kernel size */
  int32_t stride;         /* 1 or 2 */
  int32_t pad;            /* zero padding (applied AFTER pre_op, as the reference pads the activated tensor) */
  int32_t up;             /* input dilation (zero insertion) -- 2 for the dgrad of a stride-2 conv, else 1 */
  int32_t pre_op;         /* ga_pre_op applied to the input on load */
  int32_t post_act;       /* ga_act applied after bias (and before `add`) */
  const float* pre_scale; /* [cin] for GA_PRE_AFFINE_SILU (folded BN a, b) */
  const float* pre_shift;
  const void* weight;     /* SIMT: fp32 [kh*kw*cin][cout];  tensor-core: bf16 [cout][ktot] K-major */
  const float* bias;      /* [cout] or NULL */
  int32_t tf32;            /* tensor-core path only: 1 = fp32 activations + fp32 weights multiplied as TF32 (kind::tf32), else bf16 operands */
  int32_t ktot;           /* tensor-core only: row length of `weight` = kh*kw*cin (+ cin2) */
  /* per-call epilogue extras.  out = (act(acc + bias) + add) * mul;  dact_out = act'(acc + bias) */
  const void* mul;        /* optional tensor of the output's shape (backward: derivative of the producer's activation) */
  int32_t mul_dtype;      /* ga_dtype */
  int32_t mul_mode;       /* ga_mul_mode */
  void* dact_out;         /* optional: derivative of post_act at the pre-activation, saved for the backward pass */
  int32_t dact_dtype;
  int32_t act_after_add;  /* 1: out = act(acc + bias + add) (ResNet bottleneck) instead of act(acc + bias) + add */
  const float* act_slope; /* [cout] negative slopes for GA_ACT_PRELU */
  float* csum_out;        /* optional (ga_conv2d_tc only, when ga_conv2d_tc_csum_supported): per-image channel sums of the bf16 output in
                             128-pixel slices, [n][h*w/128][cout] -- exactly what ga_channel_sum would compute from the output */
} ga_conv_desc;

const char* ga_last_error(void);
/* Device-side seed salt for CUDA-graph replay: every Philox kernel uses seed + *salt when a salt buffer is registered.
 * ga_seed_salt_bump (a one-thread kernel, capturable as the first node of a graph) advances it, so each replay draws fresh noise
 * although the by-value seeds are frozen into the graph.  Pass NULL to unregister. */
int ga_seed_salt_set(uint64_t* dev_salt);
int ga_seed_salt_bump(void* stream);
/* TF32 producers: tcgen05 kind::tf32 truncates fp32 operands; while this switch is on, kernels that write fp32 ACTIVATIONS (conv_tc fp32
 * output, ga_affine_act / ga_cast to fp32, the fp32 `act` copy of ga_se_residual_fwd) round them to nearest TF32 so the truncation is exact.
 * Host-side, read at launch time on the calling thread. */
int ga_f32_round_tf32(int on);
int ga_abi_version(void);
/* number of kernels launched by this library on the calling thread since the last reset (bench.py "gpu_launches") */
int64_t ga_launch_count(int reset);

/* ---- pre-processing: abstract_models.py:129-159,173-178 (apply_gaussian_blur, add_gaussian_noise) and the
 *      NVAE input normalisation NVAE/model.py:32 -- ONE pass: blur -> + eps*noise/||noise||_2 -> clamp[0,1]
 *      -> (x-0.5)/0.5, NCHW fp32 in, NHWC out.  noise_sumsq is the per-sample reduction pre-pass. */
/* reductions are two-stage without atomics (bit-reproducible): sumsq is [n][ga_noise_sumsq_parts(chw)] partial sums */
int ga_noise_sumsq_parts(int chw);
int ga_noise_sumsq(const float* noise_nchw, int n, int chw, float* sumsq, void* stream);
int ga_noise_sumsq_philox(uint64_t seed, int64_t sample0, int n, int chw, float* sumsq, void* stream);
int ga_preprocess_fwd(const float* x_nchw, const float* noise_nchw /*NULL => philox*/, const float* sumsq,
                      uint64_t seed, int64_t sample0, float eps, const float* taps /*[2r+1] or NULL*/, int radius,
                      int normalize, const ga_tensor* out_nhwc, float* pre_nchw /*optional: value before clamp, saved for bwd*/,
                      void* stream);
/* backward of the above w.r.t. x: clamp mask, symmetric reflect-border blur transposed. g_nhwc is d/d(out). */
/* whole-image variant for 3 x 64 x 64 inputs (radius 7 or no blur): one CTA per image, image resident in shared memory, noise norm
 * reduced in-kernel -- one launch, one HBM read + one write (replaces ga_noise_sumsq* + ga_preprocess_fwd at this size) */
int ga_preprocess_image_supported(int c, int h, int w, int radius, int have_taps);
int ga_preprocess_image_fwd(const float* x_nchw, const float* noise_nchw, uint64_t seed, int64_t sample0, float eps, const float* taps,
                            int radius, int normalize, const ga_tensor* out, float* pre_nchw, void* stream);
int ga_preprocess_bwd(const ga_tensor* g_nhwc, const float* pre_nchw /*saved pre-clamp value (clamp mask)*/,
                      const float* taps, int radius, int normalize, float* tmp_nchw /*workspace, same size as gx (blur only)*/,
                      float* gx_nchw, void* stream);

/* ---- convolutions (NVAE cells: architecture.py:64-218; VGG body; linears with h=w=1) */
int ga_conv2d_simt(const ga_tensor* in, const ga_conv_desc* d, const ga_tensor* add /*nullable*/,
                   const ga_tensor* out, void* stream);
/* tcgen05/TMEM/TMA implicit GEMM, bf16 operands, fp32 accumulate.  in2: optional second K source (1x1),
 * used for the decoder combiner conv1x1(cat[x,z]) (architecture.py:205-218). out_bf16/out_f32: either or both. */
int ga_conv2d_tc(const ga_tensor* in, const ga_tensor* in2, const ga_conv_desc* d, const ga_tensor* add,
                 const ga_tensor* out_bf16, const ga_tensor* out_f32, void* stream);
int ga_conv2d_tc_supported(const ga_tensor* in, const ga_tensor* in2, const ga_conv_desc* d, int cout);
/* SE squeeze fused into the producing conv: 1 if ga_conv2d_tc (bf16 output only, no add) can also fill desc->csum_out */
int ga_conv2d_tc_csum_supported(const ga_tensor* in, const ga_conv_desc* desc, int cout);

/* depthwise 5x5, pad 2, + bias + SiLU (decoder cell, architecture.py:168-170 with BN folded).  up=1: the
 * input is read through a nearest x2 up-sampling (architecture.py:162). weight fp32 [25][c]. */
int ga_dwconv5x5_fwd(const ga_tensor* in, const float* weight, const float* bias, int act, int up,
                     const ga_tensor* out, void* stream);

/* extended form: `mul` (output's shape/dtype) multiplies the result (backward: times the saved act' of the producer),
 * `dact` receives act'(pre-activation) (taping forward).  The dgrad of the depthwise conv is the same kernel on
 * flipped taps. */
int ga_dwconv5x5_ex(const ga_tensor* in, const ga_tensor* mul, const float* weight, const float* bias, int act, int up,
                    const ga_tensor* out, const ga_tensor* dact, void* stream);

/* ---- fused decoder-cell body: r = project1x1(SiLU(dw5x5(SiLU(expand1x1(x) + be)) + dw_b)) + bp  (architecture.py:164-173, the four
 *      BatchNorms folded into the convs).  The 6C-channel hidden tensor stays in shared / tensor memory (tcgen05 + TMA).
 *      x, out: bf16 NHWC; we_tc [hidden][C], wp_tc [C][hidden] bf16 K-major; dw_w chunk-major [hidden/64][25][64] fp32.  Supported: square maps of
 *      8 / 16 / 32 pixels with C = 256 / 128 / 64 (the three decoder scales of the 64x64 NVAE); other shapes use the three kernels. */
int ga_mbconv_fused_supported(const ga_tensor* x, int hidden);
int ga_mbconv_fused(const ga_tensor* x, const void* we_tc, const float* be, const float* dw_w, const float* dw_b,
                    const void* wp_tc, const float* bp, int hidden, const ga_tensor* out, void* stream);
/* same, with two optional extras from the same pass:
 *   csum_out (or NULL): the SE squeeze of the result (architecture.py:37-61, the numerator of `x.mean(dim=[2,3])`) -- per-image channel sums of `out`
 *     as stored (bf16) in the slices ga_channel_sum uses, [N][ga_channel_sum_parts(N, H*W)][C] fp32;
 *   dact_e, dact_dw (both or neither): the tape of the attack path -- SiLU'(expand pre-activation) and SiLU'(depthwise pre-activation), bf16
 *     [N][H][W][hidden], the factors ga_conv2d_tc(mul=) / ga_dwconv5x5_ex(mul=) apply in the backward sweep (what autograd saves for
 *     architecture.py:164-173 under untargeted.py:146,201). */
int ga_mbconv_fused_ex(const ga_tensor* x, const void* we_tc, const float* be, const float* dw_w, const float* dw_b,
                       const void* wp_tc, const float* bp, int hidden, const ga_tensor* out, float* csum_out,
                       const ga_tensor* dact_e, const ga_tensor* dact_dw, void* stream);
/* input gradient of the decoder cell in ONE kernel (the attack path's backward sweep; what torch.autograd.grad computes for
 * architecture.py:164-173 under untargeted.py:146,201):   out = add + expand^T( dact_e * dw5x5^T( dact_dw * project^T(g) ) ).
 * g: bf16 NHWC gradient w.r.t. the cell body's output; wpT_tc [hidden][C], weT_tc [C][hidden]: the transposed 1x1 weights (bf16 K-major, the
 * dgrad layers' weights); dw_wT: flipped taps, chunk-major [hidden/64][25][64] fp32; dact_dw / dact_e: the tapes of ga_mbconv_fused_ex;
 * add: fp32 NHWC gradient arriving through the skip connection, or NULL; out: fp32 NHWC.  Same shapes as ga_mbconv_fused_supported. */
int ga_mbconv_fused_bwd(const ga_tensor* g, const void* wpT_tc, const float* dw_wT, const ga_tensor* dact_dw, const ga_tensor* dact_e,
                        const void* weT_tc, const ga_tensor* add, int hidden, const ga_tensor* out, void* stream);
/* debug only: per-role clock64 timeline of the 32x32 fused decoder cell; buf = device uint64[8*13*24*8] or NULL (off) */
int ga_debug_mbconv_trace(unsigned long long* buf);
/* debug only: clock64 timeline of CTA 0 of the persistent 3x3 kernel; buf = device uint64[3*16*16] or NULL (off) */
int ga_debug_c3_trace(unsigned long long* buf);
/* A/B testing: 1 = persistent halo-reuse 3x3 kernel where it applies (default), 0 = per-tap kernel everywhere */
int ga_tc_halo_enable(int on);

/* ---- squeeze-excite + residual (architecture.py:37-61,128-136,178-186) */
/* sums is [n][ga_channel_sum_parts(n, h*w)][c] partial sums (two-stage, no atomics: bit-reproducible) */
int ga_channel_sum_parts(int n, int hw);
int ga_channel_sum(const ga_tensor* r, float* sums, void* stream);
/* gate = sigmoid(W2 relu(W1 mean + b1) + b2);  out = skip + res_scale * gate * r;
 * optional extra outputs: out_bf16 copy, act = act_op(act_scale*out + act_shift) -- the next cell's BN+SiLU, or (scale/shift NULL,
 * act_op ELU) the pre-activated input of the decoder sampler / logits head (NVAE/model.py:226-231,310-313). */
int ga_se_residual_fwd(const ga_tensor* r, const float* sums, const float* w1, const float* b1, const float* w2,
                       const float* b2, int hidden, float res_scale, const ga_tensor* skip,
                       const ga_tensor* out, const ga_tensor* out2 /*nullable*/, const ga_tensor* act /*nullable*/,
                       const float* act_scale, const float* act_shift, int act_op /* GA_ACT_SILU | GA_ACT_NONE */,
                       float* gate_out /*[n][c] nullable*/, void* stream);

/* ---- per-level latent interpolation + reparameterised sampling
 *      (models.py:198-206,243-250; distributions.py:20-45).  z = (1-a)*sc(mu_p+mu_q) + a*(sc(mu_p)+eps*T*exp(sc(ls_p)))
 *      mu_q: first z channels of `q`; p: [mu_p | logsig_p] (NULL for level 0 => prior N(0,1)).
 *      eps: NCHW fp32 [n][z][h][w] or NULL => Philox stream keyed by (seed, level, global sample index). */
int ga_latent_mix_fwd(const ga_tensor* q, const ga_tensor* p /*nullable*/, const float* eps_nchw, uint64_t seed,
                      int level, int64_t sample0, const float* alpha_dev /*device scalar*/, float temperature,
                      int zdim, const ga_tensor* z_out, void* stream);

/* ---- DiscMixLogistic(...).mean() + de-normalisation (distributions.py:103-129,231-254; models.py:269-274)
 *      logits NHWC [n][h][w][10*n_mix] -> purified NCHW fp32 in [0,1] (+ optional NHWC classifier input
 *      (p-0.5)/0.5, abstract_models.py:59-60). */
int ga_discmix_mean_fwd(const ga_tensor* logits, int n_mix, float* purified_nchw, const ga_tensor* cls_in /*nullable*/,
                        void* stream);

/* ---- small layout / resampling ops */
int ga_upsample_nearest2x(const ga_tensor* in, const ga_tensor* out, void* stream);           /* architecture.py:162 */
int ga_upsample_bilinear2x(const ga_tensor* in, const ga_tensor* out, void* stream);          /* architecture.py:91 (align_corners=True) */
int ga_maxpool2x2(const ga_tensor* in, const ga_tensor* out, void* stream);                   /* torchvision vgg11_bn 'M' */
int ga_subsample2x(const ga_tensor* in, const ga_tensor* out, void* stream);                  /* nn.MaxPool2d(1, 2): encoding/helpers.py:95-96 */
int ga_maxpool3x3s2(const ga_tensor* in, const ga_tensor* out, void* stream);                 /* torchvision resnet stem pool */
int ga_global_avgpool(const ga_tensor* in, const ga_tensor* out, void* stream);               /* AdaptiveAvgPool2d(1) */
int ga_cast(const ga_tensor* in, const ga_tensor* out, void* stream);                         /* dtype cast / copy */
int ga_affine_act(const ga_tensor* in, const float* scale, const float* shift, int act, const ga_tensor* out,
                  void* stream);                                                               /* folded BN + act */
int ga_nchw_to_nhwc(const float* in_nchw, const ga_tensor* out, float scale, float shift, void* stream);

/* ---- attack inner loop: PGD-Linf step (update rule of competitors/trades/modules.py:43-45), fused
 *      x_adv <- clamp(min(max(x_adv + a*sign(g), x-eps), x+eps), 0, 1), in place, NCHW fp32 */
int ga_pgd_linf_step(float* x_adv, const float* grad, const float* x_nat, float step, float eps, int64_t numel,
                     void* stream);
/* ---- batched L2 attack steps (SURVEY 8f rank 1), one CTA per image, per-image norms, NCHW fp32 [n][chw]:
 *      APGD update of src/attacks/untargeted.py:176-193 (step along grad/||grad||, project on the L2 ball of radius `bound` around x,
 *      clamp, momentum a, project, clamp; x_adv_old <- x_adv), in place; step_size: device float[n] (per-image step sizes);
 *      FGSM update of untargeted.py:736-745 (x + l2 * sign(g)/||sign(g)||, clamp; g = gradient of +CE);
 *      APGD starting point of untargeted.py:129-131 (x + bound * noise/||noise||, clamp) */
int ga_apgd_l2_step(float* x_adv, float* x_adv_old, const float* grad, const float* x_nat, const float* step_size, float a,
                    float bound, int n, int chw, void* stream);
int ga_fgsm_l2_step(const float* x_nat, const float* grad, float l2, float* out, int n, int chw, void* stream);
int ga_l2_ball_start(const float* x_nat, const float* noise, float bound, float* out, int n, int chw, void* stream);
/* softmax cross-entropy: dlogits = (softmax - onehot)/n (mean reduction), loss[n], argmax==label counter */
int ga_softmax_xent(const float* logits, const int64_t* labels, int n, int classes, float* loss, float* dlogits,
                    int32_t* pred, unsigned long long* n_correct /*device, accumulated*/, void* stream);

/* ================================================================ StyleGAN2 generator pieces (SURVEY rows A14-A17)
 * sm_100a replacements of the reference's only native kernels (stylegan2/op/fused_bias_act_kernel.cu,
 * stylegan2/op/upfirdn2d_kernel.cu) and the glue of the modulated conv rewritten as activation scaling. */
int ga_pixelnorm(const float* x, int rows, int d, const ga_tensor* out, void* stream);                  /* generator.py:10-15 */
/* demod[n][co] = rsqrt(sum_ci s[n][ci]^2 * wsq[co][ci] + 1e-8)                                          generator.py:169-171 */
int ga_style_demod(const float* s, const float* wsq, int n, int cin, int cout, float* demod, void* stream);
int ga_channel_scale(const ga_tensor* x, const float* s /*[n][c]*/, const ga_tensor* out, void* stream); /* generator.py:164-167 */
/* v = act(y * demod[n][c] + noise_w * noise[h][w] + bias[c]) (+ skip): StyledConv / ToRGB epilogue = fused_bias_act
 * (generator.py:258-268,283-292).  phases=1: y = [n][h/2][w/2][4*c], the 4 sub-pixel phases of an up-sampling conv as channel groups.
 * out = v * scale_a[n][c], out_b = v * scale_b[n][c]: the consumers' modulation (their style vector) applied in the same pass */
int ga_styled_bias_act(const ga_tensor* y, int phases, const float* demod, const float* noise_hw, float noise_w,
                       const float* bias, int act, const ga_tensor* skip,
                       const float* skip_up_kernel /* nullable; 4x4 FIR: skip is HALF resolution and is up-sampled on the fly */,
                       const float* scale_a /*[n][c] nullable*/, const ga_tensor* out /*nullable*/, const float* scale_b,
                       const ga_tensor* out_b /*nullable*/, void* stream);
/* zero-insert up-sample -> pad -> FIR (flipped kernel) -> decimate, NHWC                                 op/upfirdn2d_kernel.cu:52-137 */
/* ToRGB in one pass (generator.py:271-292): out = conv1x1(x, w) + bias + Upsample(skip).  x: bf16 NHWC, already modulated by the layer's style;
 * w_bf16 [4][cin] (RGB padded to 4 rows); bias fp32 [4] or NULL; skip: fp32 [n][h/2][w/2][4] with its 4x4 FIR `skip_up_kernel` (upfirdn2d up 2,
 * pad (2,1)), or both NULL; out: fp32 [n][h][w][4]. */
int ga_torgb_fused(const ga_tensor* x, const void* w_bf16, const float* bias, const ga_tensor* skip, const float* skip_up_kernel,
                   const ga_tensor* out, void* stream);
int ga_upfirdn2d(const ga_tensor* in, const float* kernel, int kh, int kw, int up, int down, int pad0, int pad1,
                 const ga_tensor* out, void* stream);
int ga_avgpool_to_nchw(const ga_tensor* in, int k, int out_c, float* out_nchw, void* stream);           /* face_pool, psp.py:26,114 */
int ga_latent_lerp(const float* codes, const float* styles, const float* alphas_dev, int b, int l, int d, float* out,
                   void* stream);                                                                         /* models.py:123-124,338-339 */
/* ---- input gradient of the W+ decode (codes -> generator -> pooled image), dgrad only.  Per-(sample, channel) sums are written as
 * partials over fixed pixel slices, [n][parts][c] with parts = ga_styled_bias_act_bwd_parts(h*w, c): no atomics, the same order for a
 * sample wherever it sits in the batch.
 * Mirror of ga_styled_bias_act (+ the ToRGB 1x1 adjoint) for one styled layer, v = its taped activation act(pre) [n][h][w][c]:
 *   g_v = s_next * g_next + s_rgb * (w_rgb^T g_rgb),  g_y = g_v * lrelu'(pre) * sqrt(2) * demod  (phases=1: [n][h/2][w/2][4c], phase-major),
 *   dot_next += g_next * v,  dot_rgb += (w_rgb^T g_rgb) * v,  dot_demod += g_pre * (pre - bias - noise_w * noise) = demod * d demod.
 * g_next [n][h][w][c] fp32/bf16 or NULL; g_rgb fp32 [n][h][w][4] with w_rgb fp32 [c][4], s_rgb [n][c], or NULL; g_y NULL: dots only.
 * c = 4 * a power of two <= 1024. */
int ga_styled_bias_act_bwd_parts(int hw, int c);
int ga_styled_bias_act_bwd(const ga_tensor* v, const ga_tensor* g_next /*nullable*/, const float* s_next /*nullable*/,
                           const float* g_rgb /*nullable*/, const float* w_rgb, const float* s_rgb, const float* demod, const float* noise_hw,
                           float noise_w, const float* bias, int phases, const ga_tensor* g_y /*nullable*/, float* dot_next /*nullable*/,
                           float* dot_rgb /*nullable*/, float* dot_demod /*nullable*/, void* stream);
/* style adjoint: ds[n][c] = sum_parts dot_mod[n][.][c] - s[n][c] * sum_o (sum_parts dot_demod[n][.][o]) demod[n][o]^2 wsq[o][c]
 * (modulation term + d demod / d s, generator.py:164-171); either dot array may be NULL */
int ga_style_bwd(const float* dot_mod, int parts_mod, const float* dot_demod, int parts_demod, const float* s, const float* demod,
                 const float* wsq, int n, int cin, int cout, float* ds, void* stream);
/* adjoint of ga_latent_lerp w.r.t. the codes: g_codes[b][l] = (1 - alphas[l]) * g_out[b][l] */
int ga_latent_lerp_bwd(const float* g_out, const float* alphas_dev, int b, int l, int d, float* g_codes, void* stream);

/* ================================================================ encoder-side pieces of the StyleGAN purifiers (encoders.cu)
 * out (and optional second copy out2) = LayerNorm(x + y) * gamma + beta over the channel dim   transformer.py:54-66 (norm1-3) */
int ga_add_layernorm(const ga_tensor* x, const ga_tensor* y /*nullable*/, const float* gamma, const float* beta, float eps,
                     const ga_tensor* out, const ga_tensor* out2 /*nullable*/, void* stream);
/* multi-head attention softmax(q k^T / sqrt(dh)) v with few queries (nn.MultiheadAttention core, transformer.py:51-62):
 * q (B, Q tokens, C), k / v (B, S tokens, C'): head h reads columns [off + h*dh, off + (h+1)*dh) of its tensor, so fused
 * q|k|v or k|v projection outputs are consumed in place.  scores_ws: ga_attention_ws_floats(B, heads, Q, S) floats. */
int64_t ga_attention_ws_floats(int b, int heads, int q, int s);
int ga_attention(const ga_tensor* q, int q_off, const ga_tensor* k, int k_off, const ga_tensor* v, int v_off, int heads, int dh,
                 float* scores_ws, const ga_tensor* out, void* stream);
/* W+ codes: out[b][l] = (use_w0 && l > 0 ? heads[0][b] : 0) + heads[l][b] + latent_avg[l]   encoder.py:125-139, psp.py:92-99;
 * heads_lb = 1: heads stored [l][b][d] (map2style outputs), 0: [b][l][d] (Style-Transformer codes, models.py:318-325) */
int ga_codes_assemble(const float* heads, int heads_lb, int use_w0, const float* latent_avg /*[l][d] nullable*/, int b, int l, int d,
                      float* out, void* stream);
/* F.interpolate(mode='bilinear', align_corners=False) to (full_h, out->w), keeping rows [crop_y0, crop_y0 + out->h)
 * (kornia.geometry.resize + crop, models.py:307-308) */
int ga_resize_bilinear(const ga_tensor* in, int full_h, int crop_y0, const ga_tensor* out, void* stream);
/* generator image (N,S,S,C>=3 fp32) -> k1 x k1 face_pool -> [rows < mask_rows or >= S/k1 - mask_rows := -1 -> 2x2 mean when k2 = 2]
 * -> purified NCHW fp32 (* out_scale + out_shift = kornia denormalize) and/or the classifier's normalised NHWC input
 * (psp.py:26,114; models.py:346-351; abstract_models.py:184-185) */
int ga_image_pool_out(const ga_tensor* in, int k1, int k2, int mask_rows, float out_scale, float out_shift, float* purified_nchw,
                      const ga_tensor* cls_nhwc /*nullable*/, void* stream);
/* adjoint of ga_image_pool_out: g_img (N,S,S,4) fp32 = pooling adjoint of (g_purified * out_scale + g_cls); masked rows get zero,
 * the 4th (padding) channel is zero.  g_purified_nchw (N,3,So,So) fp32 and g_cls (N,So,So,3) may each be NULL. */
int ga_image_pool_out_bwd(const float* g_purified_nchw /*nullable*/, const ga_tensor* g_cls /*nullable*/, int k1, int k2, int mask_rows,
                          float out_scale, const ga_tensor* g_img, void* stream);
/* out[l][b][d] ~ N(0, std^2), Philox stream keyed by (seed, l, global sample index): torch.normal(0, std, (n_codes, b, d)), models.py:119,334 */
int ga_philox_codes(uint64_t seed, int64_t sample0, float std_, int l, int b, int d, float* out, void* stream);

/* ================================================================ input-gradient (dgrad-only) backward pass
 * The attacks differentiate the logits w.r.t. the input batch only (untargeted.py:146,201): weights are frozen, no
 * weight gradient is ever formed.  Conv dgrads = ga_conv2d_* on flipped/transposed weights (+ `mul` epilogue). */
/* out = g * act'(scale*x + shift) * scale (+ add): backward of the BN+SiLU / SiLU / ELU pre-activations */
int ga_affine_act_bwd(const ga_tensor* g, const ga_tensor* x, const float* scale, const float* shift, int act,
                      const ga_tensor* add /*nullable*/, const ga_tensor* out, void* stream);
int ga_add(const ga_tensor* a, const ga_tensor* b, const ga_tensor* out, void* stream);
/* backward of ga_se_residual_fwd w.r.t. r (the skip gradient is g_out itself): g_r = s*gate*g_out + d(gate MLP)/HW.
 * sums = the forward's partial channel sums of r; dots_ws = workspace of the same size. */
int ga_se_residual_bwd(const ga_tensor* g_out, const ga_tensor* r, const float* sums, float* dots_ws, const float* w1,
                       const float* b1, const float* w2, const float* b2, int hidden, float res_scale,
                       const ga_tensor* g_r, void* stream);
int ga_sumpool2x2(const ga_tensor* in, const ga_tensor* mul /*nullable, out's shape*/, const ga_tensor* out, void* stream); /* nearest x2 backward (* mul) */
int ga_upsample_bilinear2x_bwd(const ga_tensor* g_out, const ga_tensor* g_in, void* stream);
/* depth-to-space x2 (fp32): out[n][2a+pi][2b+pj][c] = in[n][a][b][(2 pi + pj) C + c] -- interleaves the four output phases of a stride-2
 * convolution's input gradient, computed as one stride-1 tensor-core conv over grad_out (replaces the zero-stuffed SIMT transposed conv;
 * reference: autograd of the stride-2 convs of architecture.py:64-82,96-136) */
int ga_depth_to_space2(const ga_tensor* in, const ga_tensor* out, void* stream);
/* gradient to the first maximal element of each window (torch semantics); relu=1 also applies the mask x_in > 0 */
int ga_maxpool2x2_bwd(const ga_tensor* x_in, const ga_tensor* g_out, int relu, const ga_tensor* g_in, void* stream);
/* ResNet / ResNeXt classifier backward (SURVEY 8f rank 3): 3x3 stride-2 pad-1 max-pool backward (first maximum wins; relu: also the ReLU
 * mask of the pooled tensor) and global-average-pool backward fused with the ReLU mask of the pooled feature map */
int ga_maxpool3x3s2_bwd(const ga_tensor* x_in, const ga_tensor* g_out, int relu, const ga_tensor* g_in, void* stream);
int ga_avgpool_bwd_relu(const ga_tensor* g_feat, const ga_tensor* y, const ga_tensor* g_in, void* stream);
int ga_latent_mix_bwd(const ga_tensor* g_z, const ga_tensor* q, const ga_tensor* p /*nullable*/, const float* eps_nchw,
                      uint64_t seed, int level, int64_t sample0, const float* alpha_dev, float temperature, int zdim,
                      const ga_tensor* g_q, const ga_tensor* g_p /*nullable*/, void* stream);
int ga_discmix_mean_bwd(const ga_tensor* logits, int n_mix, const float* g_purified_nchw /*nullable*/,
                        const ga_tensor* g_cls /*nullable*/, const ga_tensor* g_logits, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GA_B200_H */
