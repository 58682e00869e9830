// SIMT implicit-GEMM convolution (fp32 accumulate, fp32 or bf16 I/O), NHWC.
//
// This is the exact-arithmetic path: the fp32 product mode (north-star "1e-4 in fp32, identical counts")
// runs every convolution of the NVAE cells / VGG11 through it, and the bf16 mode uses it for the few layers
// the tcgen05 kernel does not take (3-channel stem convs, stride-2 cells, transposed convs of the backward).
// Replaces the cuDNN calls behind nn.Conv2d in /root/reference/src/mlvgms_autoencoders/NVAE/modules/
// architecture.py:64-218 (with weight-norm and eval-BN folded into the weights by the host).
//
// GEMM view: M = N*Ho*Wo output pixels, N = Cout, K = KH*KW*Cin.  CTA tile 128x64, K step 16, 256 threads,
// 8x4 register tile per thread, operands staged through shared memory (A transposed so the inner product
// reads float4).  Pre-op (ELU / SiLU / folded-BN+SiLU) is applied on load so the zero padding is applied to
// the *activated* tensor exactly as the reference pads after BN+SiLU (architecture.py:119-126).
#include "ga_common.cuh"

namespace ga {

constexpr int BM = 128, BN = 64, BK = 16, NT = 256;
constexpr int AS_PITCH = BM + 4;

struct ConvParams {
  const void* in;
  const float* w;
  const float* bias;
  const float* pre_scale;
  const float* pre_shift;
  const void* add;
  void* out;
  int N, H, W, Cin, Ho, Wo, Cout;
  int KH, KW, stride, pad, up;
  int pre_op, post_act;
  int add_dtype;
  const void* mul; int mul_dtype, mul_mode;
  void* dact; int dact_dtype;
  const float* act_slope; int act_after_add;
  int64_t M;
};

template <typename TIn>
__device__ __forceinline__ float load_in(const TIn* p) { return ldf<TIn>(p); }

__device__ __forceinline__ float pre_apply(float v, int pre_op, float sc, float sh) {
  switch (pre_op) {
    case GA_PRE_ELU: return eluf_(v);
    case GA_PRE_SILU: return siluf_(v);
    case GA_PRE_AFFINE_SILU: return siluf_(fmaf(v, sc, sh));
    case GA_PRE_AFFINE: return fmaf(v, sc, sh);
    default: return v;
  }
}

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(NT) conv_igemm_simt_kernel(ConvParams p) {
  __shared__ __align__(16) float As[BK][AS_PITCH];
  __shared__ __align__(16) float Bs[BK][BN];

  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const TIn* in = reinterpret_cast<const TIn*>(p.in);

  // ---- A-gather assignment: thread -> (row, 8 consecutive k)
  const int a_row = tid >> 1;
  const int a_k0 = (tid & 1) * 8;
  const int64_t a_m = m0 + a_row;
  const bool a_valid_m = a_m < p.M;
  int a_n = 0, a_oy = 0, a_ox = 0;
  if (a_valid_m) {
    int64_t t = a_m;
    a_ox = (int)(t % p.Wo); t /= p.Wo;
    a_oy = (int)(t % p.Ho); t /= p.Ho;
    a_n = (int)t;
  }
  // ---- B-load assignment: thread -> (k row, 4 consecutive n)
  const int b_k = tid >> 4;
  const int b_n = (tid & 15) * 4;
  const bool cout_vec = (p.Cout & 3) == 0;
  const bool cin_vec = (p.Cin & 7) == 0;   // 8 consecutive channels stay inside one pixel, aligned

  const int ty = tid >> 4, tx = tid & 15;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  const int Hup = (p.H - 1) * p.up + 1, Wup = (p.W - 1) * p.up + 1;   // zero-inserted extent
  const int cchunks = (p.Cin + BK - 1) / BK;

  // K loop flattened to (tap, channel chunk) steps with a register prefetch of the next step: the global loads of step
  // i+1 are in flight while step i is multiplied out of shared memory (the un-pipelined loop exposed one DRAM/L2 round
  // trip per step)
  const int steps = p.KH * p.KW * cchunks;
  float av[8], bv[4];
  auto load_step = [&](int step) {
    const int tap = step / cchunks, cc = step - tap * cchunks;
    const int ky = tap / p.KW, kx = tap - ky * p.KW;
    int iy = a_oy * p.stride - p.pad + ky;
    int ix = a_ox * p.stride - p.pad + kx;
    bool pix_ok = a_valid_m && iy >= 0 && ix >= 0 && iy < Hup && ix < Wup;
    if (p.up > 1) {
      pix_ok = pix_ok && (iy % p.up == 0) && (ix % p.up == 0);
      iy /= p.up; ix /= p.up;
    }
    const TIn* src = in + (((int64_t)a_n * p.H + iy) * p.W + ix) * p.Cin;
    const int c0 = cc * BK;
    const int ca = c0 + a_k0;
    if (pix_ok && cin_vec && ca + 8 <= p.Cin) {
      float t4[4];
      ld4<TIn>(src + ca, t4);
      av[0] = t4[0]; av[1] = t4[1]; av[2] = t4[2]; av[3] = t4[3];
      ld4<TIn>(src + ca + 4, t4);
      av[4] = t4[0]; av[5] = t4[1]; av[6] = t4[2]; av[7] = t4[3];
      if (p.pre_op != GA_PRE_NONE) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float sc = 1.f, sh = 0.f;
          if (p.pre_op >= GA_PRE_AFFINE_SILU) { sc = p.pre_scale[ca + j]; sh = p.pre_shift[ca + j]; }
          av[j] = pre_apply(av[j], p.pre_op, sc, sh);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float v = 0.0f;
        if (pix_ok && ca + j < p.Cin) {
          v = load_in<TIn>(src + ca + j);
          float sc = 1.f, sh = 0.f;
          if (p.pre_op >= GA_PRE_AFFINE_SILU) { sc = p.pre_scale[ca + j]; sh = p.pre_shift[ca + j]; }
          v = pre_apply(v, p.pre_op, sc, sh);
        }
        av[j] = v;
      }
    }
    bv[0] = bv[1] = bv[2] = bv[3] = 0.f;
    const int cb = c0 + b_k;
    if (cb < p.Cin) {
      const float* wrow = p.w + ((int64_t)tap * p.Cin + cb) * p.Cout + n0 + b_n;
      if (cout_vec && n0 + b_n + 4 <= p.Cout) {
        float4 t = *reinterpret_cast<const float4*>(wrow);
        bv[0] = t.x; bv[1] = t.y; bv[2] = t.z; bv[3] = t.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (n0 + b_n + j < p.Cout) bv[j] = wrow[j];
      }
    }
  };
  load_step(0);
  for (int step = 0; step < steps; ++step) {
    __syncthreads();   // previous tile fully consumed
#pragma unroll
    for (int j = 0; j < 8; ++j) As[a_k0 + j][a_row] = av[j];
    *reinterpret_cast<float4*>(&Bs[b_k][b_n]) = make_float4(bv[0], bv[1], bv[2], bv[3]);
    __syncthreads();
    if (step + 1 < steps) load_step(step + 1);      // prefetch: overlaps with the FMAs below
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
      float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
  }

  // ---------------- epilogue: + bias, activation, + add, store
  TOut* out = reinterpret_cast<TOut*>(p.out);
  const int nb = n0 + tx * 4;
  float bias4[4] = {0.f, 0.f, 0.f, 0.f};
  if (p.bias != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (nb + j < p.Cout) bias4[j] = p.bias[nb + j];
  }
  const bool extras = (p.mul != nullptr) || (p.dact != nullptr) || p.post_act == GA_ACT_PRELU || p.act_after_add;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = m0 + ty * 8 + i;
    if (m >= p.M) continue;
    const int64_t off = m * p.Cout + nb;
    if (extras) {                                  // backward-pass epilogues: scalar path
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (nb + j >= p.Cout) continue;
        const float pre = acc[i][j] + bias4[j];
        if (p.dact != nullptr) {
          const float dv = act_grad(pre, p.post_act);
          if (p.dact_dtype == GA_F32) reinterpret_cast<float*>(p.dact)[off + j] = dv;
          else reinterpret_cast<__nv_bfloat16*>(p.dact)[off + j] = __float2bfloat16_rn(dv);
        }
        const float slope = p.act_slope != nullptr ? p.act_slope[nb + j] : 0.f;
        float r = p.act_after_add ? pre : apply_act_s(pre, p.post_act, slope);
        if (p.add != nullptr)
          r += (p.add_dtype == GA_F32) ? reinterpret_cast<const float*>(p.add)[off + j]
                                       : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.add)[off + j]);
        if (p.act_after_add) r = apply_act_s(r, p.post_act, slope);
        if (p.mul != nullptr) {
          const float mv = (p.mul_dtype == GA_F32) ? reinterpret_cast<const float*>(p.mul)[off + j]
                                                   : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.mul)[off + j]);
          r *= mul_factor(mv, p.mul_mode, slope);
        }
        stf<TOut>(out + off + j, r);
      }
      continue;
    }
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = acc[i][j] + bias4[j];
    apply_act_n<4>(v, p.post_act);
    if (cout_vec && nb + 4 <= p.Cout) {
      if (p.add != nullptr) {
        float a4[4];
        if (p.add_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(p.add) + off, a4);
        else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(p.add) + off, a4);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] += a4[j];
      }
      st4<TOut>(out + off, v);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (nb + j >= p.Cout) continue;
        float r = v[j];
        if (p.add != nullptr) {
          r += (p.add_dtype == GA_F32) ? reinterpret_cast<const float*>(p.add)[off + j]
                                       : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.add)[off + j]);
        }
        stf<TOut>(out + off + j, r);
      }
    }
  }
}

// ---------------------------------------------------------------------------- stems: Cin <= 4, 3x3 stride 1 (NVAE init_conv 3->32,
// VGG features.0 3->64, IR-SE50 input_layer 3->64 + PReLU) and 7x7 stride 2 (torchvision ResNet conv1 3->64 + ReLU).
// K = 27 / 147 is far too short for the tiled GEMM above.  One thread owns one output pixel and ALL output channels (COUT fp32
// accumulators): every input value is loaded once, weights are broadcast from shared memory as float4 (4 FMA per LDS.128), the block
// is persistent (grid-stride over 256-pixel chunks) so the weight stage-in is paid once, and a thread's COUT outputs are one
// contiguous run of the NHWC tensor.
template <typename TIn, typename TOut, int KS, int STRIDE, int COUT>
__global__ void __launch_bounds__(256) conv_stem_kernel(const TIn* __restrict__ in, const float* __restrict__ w, const float* __restrict__ bias,
                                                        const float* __restrict__ slope, int post_act, int N, int H, int W, int Cin, int Ho,
                                                        int Wo, TOut* __restrict__ out) {
  extern __shared__ float s_w[];                      // [KS*KS*Cin][COUT] | bias[COUT] | slope[COUT]
  constexpr int PAD = KS / 2;
  const int K = KS * KS * Cin;
  for (int i = threadIdx.x; i < K * COUT; i += 256) s_w[i] = w[i];
  for (int i = threadIdx.x; i < COUT; i += 256) {
    s_w[K * COUT + i] = bias ? bias[i] : 0.f;
    s_w[(K + 1) * COUT + i] = slope ? slope[i] : 0.f;
  }
  __syncthreads();
  const int64_t total_pix = (int64_t)N * Ho * Wo;
  for (int64_t pix = (int64_t)blockIdx.x * 256 + threadIdx.x; pix < total_pix; pix += (int64_t)gridDim.x * 256) {
    const int x = (int)(pix % Wo);
    const int y = (int)((pix / Wo) % Ho);
    const int64_t n = pix / ((int64_t)Wo * Ho);
    float acc[COUT];
#pragma unroll
    for (int j = 0; j < COUT; ++j) acc[j] = s_w[K * COUT + j];
#pragma unroll 1
    for (int ky = 0; ky < KS; ++ky) {
      const int iy = y * STRIDE + ky - PAD;
      if (iy < 0 || iy >= H) continue;
#pragma unroll 1
      for (int kx = 0; kx < KS; ++kx) {
        const int ix = x * STRIDE + kx - PAD;
        if (ix < 0 || ix >= W) continue;
        const TIn* src = in + ((n * H + iy) * W + ix) * Cin;
        const float* wk = s_w + (ky * KS + kx) * Cin * COUT;
        for (int ci = 0; ci < Cin; ++ci) {
          const float v = ldf<TIn>(src + ci);
#pragma unroll
          for (int j = 0; j < COUT; j += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(wk + ci * COUT + j);
            acc[j] = fmaf(v, w4.x, acc[j]); acc[j + 1] = fmaf(v, w4.y, acc[j + 1]);
            acc[j + 2] = fmaf(v, w4.z, acc[j + 2]); acc[j + 3] = fmaf(v, w4.w, acc[j + 3]);
          }
        }
      }
    }
    if (post_act == GA_ACT_PRELU) {
#pragma unroll
      for (int j = 0; j < COUT; ++j) acc[j] = acc[j] > 0.f ? acc[j] : s_w[(K + 1) * COUT + j] * acc[j];
    } else {
      apply_act_n<COUT>(acc, post_act);
    }
    TOut* dst = out + pix * COUT;
#pragma unroll
    for (int j = 0; j < COUT; j += 4) {
      const float o[4] = {acc[j], acc[j + 1], acc[j + 2], acc[j + 3]};
      st4<TOut>(dst + j, o);
    }
  }
}

template <typename TIn, typename TOut, int KS, int STRIDE, int COUT>
static int launch_stem_t(const ga_tensor* in, const ga_conv_desc* d, const ga_tensor* out, cudaStream_t s) {
  const int K = KS * KS * in->c;
  const int64_t total_pix = (int64_t)out->n * out->h * out->w;
  const size_t smem = (size_t)(K + 2) * COUT * sizeof(float);
  static bool configured = false;
  if (!configured && smem > 48 * 1024) {
    GA_CUDA(cudaFuncSetAttribute(conv_stem_kernel<TIn, TOut, KS, STRIDE, COUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  int sms = 148;
  const int64_t want = (total_pix + 255) / 256;
  const int grid = (int)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);       // persistent: <= 8 blocks per SM
  conv_stem_kernel<TIn, TOut, KS, STRIDE, COUT><<<grid, 256, smem, s>>>((const TIn*)in->data, (const float*)d->weight, d->bias, d->act_slope,
                                                                       d->post_act, in->n, in->h, in->w, in->c, out->h, out->w,
                                                                       (TOut*)out->data);
  GA_LAUNCH_OK();
  return 0;
}

template <typename TIn, typename TOut>
static int launch_stem(const ga_tensor* in, const ga_conv_desc* d, const ga_tensor* out, cudaStream_t s) {
  if (d->kh == 3 && d->stride == 1) {
    if (out->c == 32) return launch_stem_t<TIn, TOut, 3, 1, 32>(in, d, out, s);
    if (out->c == 64) return launch_stem_t<TIn, TOut, 3, 1, 64>(in, d, out, s);
  }
  if (d->kh == 7 && d->stride == 2 && out->c == 64) return launch_stem_t<TIn, TOut, 7, 2, 64>(in, d, out, s);
  return -1;     // not a stem shape
}

static bool is_stem(const ga_tensor* in, const ga_conv_desc* d, const ga_tensor* add, const ga_tensor* out) {
  if (in->c > 4 || d->up != 1 || d->pre_op != GA_PRE_NONE || add != nullptr || d->mul != nullptr || d->dact_out != nullptr ||
      d->act_after_add || numel(out) == 0 || d->kh != d->kw)
    return false;
  if (d->kh == 3 && d->stride == 1 && d->pad == 1) return out->c == 32 || out->c == 64;
  return d->kh == 7 && d->stride == 2 && d->pad == 3 && out->c == 64;
}

}  // namespace ga

extern "C" int ga_conv2d_simt(const ga_tensor* in, const ga_conv_desc* d, const ga_tensor* add, const ga_tensor* out,
                              void* stream) {
  using namespace ga;
  GA_CHECK(in && d && out, "ga_conv2d_simt: null argument");
  GA_CHECK(d->stride >= 1 && d->up >= 1 && d->kh >= 1 && d->kw >= 1, "ga_conv2d_simt: bad geometry");
  GA_CHECK(!(d->stride > 1 && d->up > 1), "ga_conv2d_simt: stride and up are exclusive");
  const int Hup = (in->h - 1) * d->up + 1, Wup = (in->w - 1) * d->up + 1;
  const int Ho = (Hup + 2 * d->pad - d->kh) / d->stride + 1;
  const int Wo = (Wup + 2 * d->pad - d->kw) / d->stride + 1;
  // transposed convs may request one extra row/col (output_padding); accept out->h in {Ho, Ho+1}
  GA_CHECK(out->n == in->n && (out->h == Ho || (d->up > 1 && out->h == Ho + 1)) &&
               (out->w == Wo || (d->up > 1 && out->w == Wo + 1)),
           "ga_conv2d_simt: output shape (%d,%d,%d) does not match conv geometry (%d,%d,%d)", out->n, out->h, out->w,
           in->n, Ho, Wo);
  GA_CHECK(d->pre_op < GA_PRE_AFFINE_SILU || (d->pre_scale && d->pre_shift), "ga_conv2d_simt: affine pre-op needs scale/shift");
  if (add) GA_CHECK(same_shape(add, out), "ga_conv2d_simt: add shape mismatch");
  // stem fast path: Cin <= 4, 3x3 stride 1 or 7x7 stride 2, no extras
  if (is_stem(in, d, add, out)) {
    cudaStream_t s = (cudaStream_t)stream;
    GA_CHECK(d->post_act != GA_ACT_PRELU || d->act_slope != nullptr, "ga_conv2d_simt: PReLU needs act_slope");
    if (in->dtype == GA_F32 && out->dtype == GA_F32) return launch_stem<float, float>(in, d, out, s);
    if (in->dtype == GA_BF16 && out->dtype == GA_BF16) return launch_stem<__nv_bfloat16, __nv_bfloat16>(in, d, out, s);
    if (in->dtype == GA_BF16 && out->dtype == GA_F32) return launch_stem<__nv_bfloat16, float>(in, d, out, s);
    return launch_stem<float, __nv_bfloat16>(in, d, out, s);
  }
  ConvParams p;
  p.in = in->data; p.w = (const float*)d->weight; p.bias = d->bias;
  p.pre_scale = d->pre_scale; p.pre_shift = d->pre_shift;
  p.add = add ? add->data : nullptr; p.add_dtype = add ? add->dtype : GA_F32;
  p.mul = d->mul; p.mul_dtype = d->mul_dtype; p.mul_mode = d->mul_mode;
  p.dact = d->dact_out; p.dact_dtype = d->dact_dtype;
  p.act_slope = d->act_slope; p.act_after_add = d->act_after_add;
  GA_CHECK(d->post_act != GA_ACT_PRELU || d->act_slope != nullptr, "ga_conv2d_simt: PReLU needs act_slope");
  GA_CHECK(d->mul == nullptr || d->mul_mode != GA_MUL_PRELU_FROM_Y || d->act_slope != nullptr, "ga_conv2d_simt: PReLU mask needs act_slope");
  p.out = out->data;
  p.N = in->n; p.H = in->h; p.W = in->w; p.Cin = in->c; p.Ho = out->h; p.Wo = out->w; p.Cout = out->c;
  p.KH = d->kh; p.KW = d->kw; p.stride = d->stride; p.pad = d->pad; p.up = d->up;
  p.pre_op = d->pre_op; p.post_act = d->post_act;
  p.M = (int64_t)out->n * out->h * out->w;
  if (p.M == 0 || p.Cout == 0) return 0;
  dim3 grid(cdiv(p.M, BM), cdiv(p.Cout, BN));
  cudaStream_t s = (cudaStream_t)stream;
  if (in->dtype == GA_F32 && out->dtype == GA_F32) conv_igemm_simt_kernel<float, float><<<grid, NT, 0, s>>>(p);
  else if (in->dtype == GA_BF16 && out->dtype == GA_BF16) conv_igemm_simt_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, NT, 0, s>>>(p);
  else if (in->dtype == GA_BF16 && out->dtype == GA_F32) conv_igemm_simt_kernel<__nv_bfloat16, float><<<grid, NT, 0, s>>>(p);
  else conv_igemm_simt_kernel<float, __nv_bfloat16><<<grid, NT, 0, s>>>(p);
  GA_LAUNCH_OK();
  return 0;
}
