// StyleGAN2 generator pieces (E4E / Style-Transformer decoders, SURVEY rows A14-A17): sm_100a replacements of the
// reference's only native kernels -- `fused_bias_act` (stylegan2/op/fused_bias_act_kernel.cu:19-49) and `upfirdn2d`
// (stylegan2/op/upfirdn2d_kernel.cu:52-137) -- plus the elementwise glue of the modulated convolution rewritten as
// "scale input channels by the style -> ONE shared-weight dense conv (tcgen05 kernel) -> scale output channels by the
// demodulation" (exact, SURVEY Appendix D; the reference materialises B x weight copies and runs a grouped conv with
// groups = B, stylegan2/generator.py:163-207).  All kernels are HBM-bound, NHWC, vectorised along channels.
#include <stdlib.h>
#include "ga_common.cuh"

namespace ga {

__device__ __forceinline__ float ld1s(const void* base, int dtype, int64_t off) {
  return dtype == GA_F32 ? reinterpret_cast<const float*>(base)[off]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[off]);
}
__device__ __forceinline__ void st1s(void* base, int dtype, int64_t off, float v) {
  if (dtype == GA_F32) reinterpret_cast<float*>(base)[off] = v;
  else reinterpret_cast<__nv_bfloat16*>(base)[off] = __float2bfloat16_rn(v);
}
__device__ __forceinline__ void ld4s(const void* base, int dtype, int64_t off, float (&v)[4]) {
  if (dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(base) + off, v);
  else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(base) + off, v);
}
__device__ __forceinline__ void st4s(void* base, int dtype, int64_t off, const float (&v)[4]) {
  if (dtype == GA_F32) st4<float>(reinterpret_cast<float*>(base) + off, v);
  else st4<__nv_bfloat16>(reinterpret_cast<__nv_bfloat16*>(base) + off, v);
}

// ---------------------------------------------------------------------------- PixelNorm (generator.py:10-15): one warp per row
__global__ void pixelnorm_kernel(const float* __restrict__ x, int rows, int d, void* out, int out_dtype) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (int64_t)row * d;
  float s = 0.f;
  for (int i = lane; i < d; i += 32) s = fmaf(xr[i], xr[i], s);
  s = warp_sum(s);
  const float r = rsqrtf(s / (float)d + 1e-8f);
  for (int i = lane; i < d; i += 32) st1s(out, out_dtype, (int64_t)row * d + i, xr[i] * r);
}

// ---------------------------------------------------------------------------- demodulation factors (generator.py:169-171)
// demod[n, co] = rsqrt( sum_ci s[n,ci]^2 * wsq[co,ci] + 1e-8 ),  wsq[co,ci] = sum_k (scale * W[co,ci,k])^2
__global__ void style_demod_kernel(const float* __restrict__ s, const float* __restrict__ wsq, int N, int Cin, int Cout,
                                   float* __restrict__ demod) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= N * Cout) return;
  const int n = w / Cout, co = w % Cout;
  float a = 0.f;
  for (int ci = lane; ci < Cin; ci += 32) {
    const float sv = s[(int64_t)n * Cin + ci];
    a = fmaf(sv * sv, wsq[(int64_t)co * Cin + ci], a);
  }
  a = warp_sum(a);
  if (lane == 0) demod[(int64_t)n * Cout + co] = rsqrtf(a + 1e-8f);
}

// ---------------------------------------------------------------------------- x[n,p,c] * s[n,c]  (modulation as activation scaling)
__global__ void __launch_bounds__(256) channel_scale_kernel(const void* x, int x_dtype, const float* __restrict__ s, int HW, int C,
                                                            int64_t total4, void* out, int out_dtype) {
  const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const int64_t i = i4 * 4;
  const int c = (int)(i % C);
  const int64_t n = i / ((int64_t)HW * C);
  float v[4];
  ld4s(x, x_dtype, i, v);
  const float4 sc = __ldg(reinterpret_cast<const float4*>(s + n * C + c));
  v[0] *= sc.x; v[1] *= sc.y; v[2] *= sc.z; v[3] *= sc.w;
  st4s(out, out_dtype, i, v);
}

// ---------------------------------------------------------------------------- fused demod + noise + bias + leaky-ReLU*sqrt(2)
// out[n,y,x,c] = act( y_conv * demod[n,c] + noise_w * noise[y,x] + bias[c] ) (+ skip)    -- StyledConv.forward (generator.py:258-268)
// and ToRGB (generator.py:283-292, act = none, demod = NULL, skip = up-sampled RGB).  This is the `fused_bias_act` equivalent.
// phases = 1: y_conv = [N][H/2][W/2][4*C], the 4 sub-pixel phases of an up-sampling conv as channel groups (see stylegan_engine.py).
__global__ void __launch_bounds__(256) styled_bias_act_kernel(const void* y, int y_dtype, int phases, const float* __restrict__ demod,
                                                              const float* __restrict__ noise, float noise_w,
                                                              const float* __restrict__ bias, int act, const void* skip, int skip_dtype,
                                                              int N, int H, int W, int C, const float* __restrict__ scale_a, void* out,
                                                              int out_dtype, const float* __restrict__ scale_b, void* out_b, int out_b_dtype,
                                                              const float* __restrict__ skip_up_kernel) {
  const int c4n = C >> 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * H * W * c4n) return;
  const int c = (int)(idx % c4n) * 4;
  int64_t t = idx / c4n;
  const int x = (int)(t % W); t /= W;
  const int yy = (int)(t % H);
  const int64_t n = t / H;
  int64_t src;
  if (phases) {
    // the four sub-pixel phases of the up-sampling conv are channel groups [ph*C, (ph+1)*C) of ONE half-resolution conv output
    const int ph = (yy & 1) * 2 + (x & 1);
    const int Hh = H >> 1, Wh = W >> 1;
    src = (((n * Hh + (yy >> 1)) * Wh + (x >> 1)) * 4 + ph) * C + c;
  } else {
    src = ((n * H + yy) * W + x) * C + c;
  }
  float v[4];
  ld4s(y, y_dtype, src, v);
  if (demod != nullptr) {
    const float4 d = __ldg(reinterpret_cast<const float4*>(demod + n * C + c));
    v[0] *= d.x; v[1] *= d.y; v[2] *= d.z; v[3] *= d.w;
  }
  const float nz = noise != nullptr ? noise_w * __ldg(noise + (int64_t)yy * W + x) : 0.f;
  float b4[4] = {0.f, 0.f, 0.f, 0.f};
  if (bias != nullptr) { const float4 b = __ldg(reinterpret_cast<const float4*>(bias + c)); b4[0] = b.x; b4[1] = b.y; b4[2] = b.z; b4[3] = b.w; }
  const int64_t o = ((n * H + yy) * W + x) * C + c;
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = v[j] + nz + b4[j];
  apply_act_n<4>(v, act);
  if (skip != nullptr && skip_up_kernel == nullptr) {
    float s4[4];
    ld4s(skip, skip_dtype, o, s4);
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] += s4[j];
  } else if (skip != nullptr) {
    // `skip` is the HALF-resolution RGB image: its `Upsample` (upfirdn2d, up 2, 4x4 FIR, pad (2,1); generator.py:28-47) is evaluated
    // here -- 4 of the 16 taps hit non-inserted samples -- instead of materialising the up-sampled image in HBM
    const int Hs = H >> 1, Ws = W >> 1;
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const int uy = yy + ky - 2;
      if (uy < 0 || uy >= H || (uy & 1)) continue;
#pragma unroll
      for (int kx = 0; kx < 4; ++kx) {
        const int ux = x + kx - 2;
        if (ux < 0 || ux >= W || (ux & 1)) continue;
        float s4[4];
        ld4s(skip, skip_dtype, ((n * Hs + (uy >> 1)) * Ws + (ux >> 1)) * C + c, s4);
        const float kw = __ldg(skip_up_kernel + (3 - ky) * 4 + (3 - kx));
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = fmaf(s4[j], kw, v[j]);
      }
    }
  }
  // the consumers are modulated convs: their per-sample input scaling (the "modulation", generator.py:164-167) is applied here on the
  // fp32 value, so no separate scaling pass (and no second bf16 rounding) exists -- one copy per consumer (next StyledConv / ToRGB)
  if (out_b != nullptr) {
    const float4 sb = __ldg(reinterpret_cast<const float4*>(scale_b + n * C + c));
    const float w[4] = {v[0] * sb.x, v[1] * sb.y, v[2] * sb.z, v[3] * sb.w};
    st4s(out_b, out_b_dtype, o, w);
  }
  if (out != nullptr) {
    if (scale_a != nullptr) {
      const float4 sa = __ldg(reinterpret_cast<const float4*>(scale_a + n * C + c));
      v[0] *= sa.x; v[1] *= sa.y; v[2] *= sa.z; v[3] *= sa.w;
    }
    st4s(out, out_dtype, o, v);
  }
}

// Fast path of the same op for the generator's big layers (bf16 outputs, lrelu * sqrt(2), no skip, power-of-two H / W / C/8): 8 channels
// (16 bytes) per item, 4 items per thread with all loads issued before the first store, 32-bit index math (shifts and masks instead of the
// 64-bit divisions of the general kernel, which ran at 1.8 TB/s = 28% of the HBM peak on the 1024^2 layers).
struct SbaFast {
  const void* y; const float* demod; const float* noise; const float* bias; const float* scale_a; const float* scale_b;
  __nv_bfloat16* out; __nv_bfloat16* out_b;
  float noise_w;
  int lw, lh, lc8;            // log2 of W, H, C/8
  uint32_t total;             // 8-channel items
};

template <bool PHASES, bool Y_F32>
__global__ void __launch_bounds__(256) styled_bias_act_vec8_kernel(const SbaFast p) {
  constexpr int U = 4;
  const uint32_t W = 1u << p.lw, H = 1u << p.lh, c8n = 1u << p.lc8, C = c8n * 8;
  const uint32_t v0 = blockIdx.x * (256u * U) + threadIdx.x;
  uint4 raw[U][Y_F32 ? 2 : 1];
  uint32_t oidx[U], nn[U], cc[U];
  float nz[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const uint32_t v = v0 + u * 256u;
    oidx[u] = 0xffffffffu;
    if (v >= p.total) continue;
    const uint32_t c8 = v & (c8n - 1), pix = v >> p.lc8;
    const uint32_t x = pix & (W - 1), yy = (pix >> p.lw) & (H - 1), n = pix >> (p.lw + p.lh);
    uint64_t src;
    if (PHASES) {
      const uint32_t ph = (yy & 1) * 2 + (x & 1);
      src = ((((uint64_t)n << (p.lh - 1)) + (yy >> 1) << (p.lw - 1)) + (x >> 1)) * (4ull * C) + ph * C + c8 * 8;
    } else {
      src = (uint64_t)v * 8;
    }
    if (Y_F32) {
      const uint4* q = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.y) + src);
      raw[u][0] = __ldg(q); raw[u][Y_F32 ? 1 : 0] = __ldg(q + 1);
    } else {
      raw[u][0] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.y) + src));
    }
    oidx[u] = v; nn[u] = n; cc[u] = c8 * 8;
    nz[u] = p.noise != nullptr ? p.noise_w * __ldg(p.noise + (pix & ((1u << (p.lw + p.lh)) - 1))) : 0.f;
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (oidx[u] == 0xffffffffu) continue;
    float v[8];
    if (Y_F32) {
      const uint4 a = raw[u][0], b = raw[u][Y_F32 ? 1 : 0];
      v[0] = __uint_as_float(a.x); v[1] = __uint_as_float(a.y); v[2] = __uint_as_float(a.z); v[3] = __uint_as_float(a.w);
      v[4] = __uint_as_float(b.x); v[5] = __uint_as_float(b.y); v[6] = __uint_as_float(b.z); v[7] = __uint_as_float(b.w);
    } else {
      const uint32_t w[4] = {raw[u][0].x, raw[u][0].y, raw[u][0].z, raw[u][0].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) { v[2 * j] = __uint_as_float(w[j] << 16); v[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u); }
    }
    const uint32_t pc = nn[u] * C + cc[u];
    if (p.demod != nullptr) {
      const float4 d0 = __ldg(reinterpret_cast<const float4*>(p.demod + pc)), d1 = __ldg(reinterpret_cast<const float4*>(p.demod + pc + 4));
      v[0] *= d0.x; v[1] *= d0.y; v[2] *= d0.z; v[3] *= d0.w; v[4] *= d1.x; v[5] *= d1.y; v[6] *= d1.z; v[7] *= d1.w;
    }
    float b8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (p.bias != nullptr) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + cc[u])), b1 = __ldg(reinterpret_cast<const float4*>(p.bias + cc[u] + 4));
      b8[0] = b0.x; b8[1] = b0.y; b8[2] = b0.z; b8[3] = b0.w; b8[4] = b1.x; b8[5] = b1.y; b8[6] = b1.z; b8[7] = b1.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float t = v[j] + nz[u] + b8[j];                       // same association as the general kernel: (y * demod + noise) + bias
      v[j] = (t > 0.0f ? t : 0.2f * t) * 1.4142135623730951f;
    }
    const uint64_t o = (uint64_t)oidx[u] * 8;
    if (p.out_b != nullptr) {
      const float4 s0 = __ldg(reinterpret_cast<const float4*>(p.scale_b + pc)), s1 = __ldg(reinterpret_cast<const float4*>(p.scale_b + pc + 4));
      *reinterpret_cast<uint4*>(p.out_b + o) = make_uint4(pack_bf16x2(v[0] * s0.x, v[1] * s0.y), pack_bf16x2(v[2] * s0.z, v[3] * s0.w),
                                                          pack_bf16x2(v[4] * s1.x, v[5] * s1.y), pack_bf16x2(v[6] * s1.z, v[7] * s1.w));
    }
    if (p.out != nullptr) {
      if (p.scale_a != nullptr) {
        const float4 s0 = __ldg(reinterpret_cast<const float4*>(p.scale_a + pc)), s1 = __ldg(reinterpret_cast<const float4*>(p.scale_a + pc + 4));
        v[0] *= s0.x; v[1] *= s0.y; v[2] *= s0.z; v[3] *= s0.w; v[4] *= s1.x; v[5] *= s1.y; v[6] *= s1.z; v[7] *= s1.w;
      }
      *reinterpret_cast<uint4*>(p.out + o) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    }
  }
}

// ---------------------------------------------------------------------------- ToRGB in one pass (generator.py:271-292)
// out[n,y,x,j] = sum_c x[n,y,x,c] * w[j][c] + bias[j] + Upsample(skip)[n,y,x,j]      (x already modulated by the layer's style, no demodulation)
// The 1x1 conv to 3 (padded 4) channels is a 64-byte-per-pixel dot product: on the tensor-core kernel it ran at 1.25 TB/s (a 128-pixel tile per CTA
// for 4 output columns), followed by a second pass for bias + skip.  Here: one thread per pixel, 16-byte loads, weights broadcast from shared
// memory, the half-resolution skip up-sampled on the fly (4 of the 16 FIR taps hit real samples), one float4 store.
__global__ void __launch_bounds__(256) torgb_fused_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                                          const float* __restrict__ bias, const float* __restrict__ skip,
                                                          const float* __restrict__ upk, int N, int H, int W, int cin,
                                                          float* __restrict__ out) {
  extern __shared__ float4 s_w[];                 // [cin]: the 4 output weights of input channel c
  for (int c = threadIdx.x; c < cin; c += 256)
    s_w[c] = make_float4(__bfloat162float(w[c]), __bfloat162float(w[cin + c]), __bfloat162float(w[2 * cin + c]), __bfloat162float(w[3 * cin + c]));
  __syncthreads();
  const int64_t pix = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (pix >= (int64_t)N * H * W) return;
  const uint4* xp = reinterpret_cast<const uint4*>(x + pix * cin);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (int c8 = 0; c8 < cin; c8 += 32) {          // 4 vectors (32 channels) in flight per trip
    uint4 v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = (c8 + 8 * i < cin) ? __ldg(xp + (c8 >> 3) + i) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (c8 + 8 * i >= cin) break;
      const uint32_t q[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float lo = __uint_as_float(q[j] << 16), hi = __uint_as_float(q[j] & 0xffff0000u);
        const float4 w0 = s_w[c8 + 8 * i + 2 * j], w1 = s_w[c8 + 8 * i + 2 * j + 1];
        a0 = fmaf(lo, w0.x, a0); a1 = fmaf(lo, w0.y, a1); a2 = fmaf(lo, w0.z, a2); a3 = fmaf(lo, w0.w, a3);
        a0 = fmaf(hi, w1.x, a0); a1 = fmaf(hi, w1.y, a1); a2 = fmaf(hi, w1.z, a2); a3 = fmaf(hi, w1.w, a3);
      }
    }
  }
  if (bias != nullptr) { const float4 b = __ldg(reinterpret_cast<const float4*>(bias)); a0 += b.x; a1 += b.y; a2 += b.z; a3 += b.w; }
  if (skip != nullptr) {
    const int xx = (int)(pix % W);
    const int64_t t = pix / W;
    const int yy = (int)(t % H);
    const int64_t n = t / H;
    const int Hs = H >> 1, Ws = W >> 1;
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const int uy = yy + ky - 2;
      if (uy < 0 || uy >= H || (uy & 1)) continue;
#pragma unroll
      for (int kx = 0; kx < 4; ++kx) {
        const int ux = xx + kx - 2;
        if (ux < 0 || ux >= W || (ux & 1)) continue;
        const float4 sv = __ldg(reinterpret_cast<const float4*>(skip + ((n * Hs + (uy >> 1)) * Ws + (ux >> 1)) * 4));
        const float kw = __ldg(upk + (3 - ky) * 4 + (3 - kx));
        a0 = fmaf(sv.x, kw, a0); a1 = fmaf(sv.y, kw, a1); a2 = fmaf(sv.z, kw, a2); a3 = fmaf(sv.w, kw, a3);
      }
    }
  }
  *reinterpret_cast<float4*>(out + pix * 4) = make_float4(a0, a1, a2, a3);
}

static int ilog2_exact(int v) {
  if (v <= 0 || (v & (v - 1))) return -1;
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

// ---------------------------------------------------------------------------- upfirdn2d (general; op/upfirdn2d_kernel.cu:52-137)
// out[o] = sum_k U[o*down + k - pad0] * kernel[K-1-k],  U = zero-insertion up-sampling of the input (per dimension)
__global__ void upfirdn2d_kernel(const void* in, int in_dtype, const float* __restrict__ kern, int KH, int KW, int up, int down, int pad0,
                                 int N, int H, int W, int C, int Ho, int Wo, void* out, int out_dtype) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * C) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int ox = (int)(t % Wo); t /= Wo;
  const int oy = (int)(t % Ho);
  const int64_t n = t / Ho;
  float acc = 0.f;
  for (int ky = 0; ky < KH; ++ky) {
    const int uy = oy * down + ky - pad0;
    if (uy < 0 || uy >= H * up || (uy % up) != 0) continue;
    const int iy = uy / up;
    for (int kx = 0; kx < KW; ++kx) {
      const int ux = ox * down + kx - pad0;
      if (ux < 0 || ux >= W * up || (ux % up) != 0) continue;
      const int ix = ux / up;
      acc = fmaf(ld1s(in, in_dtype, ((n * H + iy) * W + ix) * C + c), kern[(KH - 1 - ky) * KW + (KW - 1 - kx)], acc);
    }
  }
  st1s(out, out_dtype, idx, acc);
}

// ---------------------------------------------------------------------------- k x k mean pooling (face_pool, psp.py:26,114), NHWC in -> NCHW fp32 out
__global__ void avgpool_to_nchw_kernel(const void* in, int in_dtype, int N, int H, int W, int C, int Co, int k, float* __restrict__ out) {
  const int Ho = H / k, Wo = W / k;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;          // over NCHW output (Co <= C channels kept)
  if (idx >= (int64_t)N * Co * Ho * Wo) return;
  const int ox = (int)(idx % Wo);
  int64_t t = idx / Wo;
  const int oy = (int)(t % Ho); t /= Ho;
  const int c = (int)(t % Co);
  const int64_t n = t / Co;
  float acc = 0.f;
  for (int dy = 0; dy < k; ++dy)
    for (int dx = 0; dx < k; ++dx) acc += ld1s(in, in_dtype, ((n * H + oy * k + dy) * W + ox * k + dx) * C + c);
  out[idx] = acc / (float)(k * k);
}

// ---------------------------------------------------------------------------- per-level latent interpolation of the W+ codes
// out[b,l,:] = (1 - a_l) * codes[b,l,:] + a_l * styles[b,l,:]      (models.py:123-124, 338-339)
__global__ void latent_lerp_kernel(const float* __restrict__ codes, const float* __restrict__ styles, const float* __restrict__ alphas,
                                   int L, int D, int64_t total, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float a = alphas[(i / D) % L];
  out[i] = (1.f - a) * codes[i] + a * styles[i];
}

// ============================================================================ input-gradient backward of the generator (W+ decode half)
// Partial per-(sample, channel) sums over FIXED pixel slices: a slice holds ~32K elements whatever the batch, so every reduction runs
// in the same order for a sample wherever it sits in the batch (bit-reproducible, no atomics; DESIGN §3).
static int sba_bwd_pix_per_part(int c) { return c >= 32768 ? 1 : 32768 / c; }

struct SbaBwd {
  const void* v; int v_dtype;                          // taped activation act(pre) [n][h][w][c]
  const void* g_next; int g_next_dtype;                // gradient w.r.t. the next conv's (modulated) input [n][h][w][c], nullable
  const float* s_next;                                 // [n][c] the next conv's style, nullable
  const float* g_rgb; const float* w_rgb;              // ToRGB output gradient [n][h][w][4] fp32 and its weights [c][4] fp32, nullable
  const float* s_rgb;                                  // [n][c]
  const float* demod; const float* noise; float noise_w; const float* bias;
  void* g_y; int g_y_dtype; int phases;                // conv-output gradient, nullable (dots only)
  float* dot_next; float* dot_rgb; float* dot_demod;   // [n][parts][c], nullable
  int H, W, C, ppp, parts;
};

// Mirror of styled_bias_act (+ the 1x1 ToRGB adjoint of torgb_fused) for one styled layer, one pass:
//   g_v   = s_next * g_next + s_rgb * (W_rgb^T g_rgb)
//   g_pre = g_v * lrelu'(pre) * sqrt(2)                 (sign of the taped activation = sign of pre)
//   g_y   = g_pre * demod                               (phase-major [n][h/2][w/2][4c] for up-sampling layers)
//   dots:  sum g_next * v (d s_next),  sum (W_rgb^T g_rgb) * v (d s_rgb),  sum g_pre * u = demod * d demod,  u = pre - bias - noise,
//          pre recovered by inverting the leaky ReLU of v (no division by demod or s).
// grid (parts, n); thread = (4-channel group, pixel lane); lanes reduce through shared memory in a fixed order.
__global__ void __launch_bounds__(256) styled_bias_act_bwd_kernel(const SbaBwd p) {
  extern __shared__ float sm[];                        // [C][4] ToRGB weights, then 3 x [256][4] partial sums
  float4* s_w = reinterpret_cast<float4*>(sm);
  float* red = sm + (p.w_rgb != nullptr ? p.C * 4 : 0);
  if (p.w_rgb != nullptr)
    for (int c = threadIdx.x; c < p.C; c += 256) s_w[c] = __ldg(reinterpret_cast<const float4*>(p.w_rgb) + c);
  __syncthreads();
  const int c4n = p.C >> 2, lanes = 256 / c4n;
  const int cg = threadIdx.x % c4n, lane = threadIdx.x / c4n, c = cg * 4;
  const int part = blockIdx.x;
  const int64_t n = blockIdx.y;
  const int HW = p.H * p.W;
  const int p0 = part * p.ppp, p1 = min(HW, p0 + p.ppp);
  const float kpos = 1.4142135623730951f, kneg = 0.2f * 1.4142135623730951f;
  float sn[4] = {0.f, 0.f, 0.f, 0.f}, sr[4] = {0.f, 0.f, 0.f, 0.f}, dm[4] = {1.f, 1.f, 1.f, 1.f}, bs[4] = {0.f, 0.f, 0.f, 0.f};
  for (int j = 0; j < 4; ++j) {
    if (p.s_next) sn[j] = p.s_next[n * p.C + c + j];
    if (p.g_rgb) sr[j] = p.s_rgb[n * p.C + c + j];
    if (p.demod) dm[j] = p.demod[n * p.C + c + j];
    if (p.bias) bs[j] = p.bias[c + j];
  }
  float a_next[4] = {0.f, 0.f, 0.f, 0.f}, a_rgb[4] = {0.f, 0.f, 0.f, 0.f}, a_dem[4] = {0.f, 0.f, 0.f, 0.f};
  for (int pix = p0 + lane; pix < p1; pix += lanes) {
    const int64_t o = (n * HW + pix) * p.C + c;
    float v[4], gv[4] = {0.f, 0.f, 0.f, 0.f};
    ld4s(p.v, p.v_dtype, o, v);
    if (p.g_next) {
      float gn[4];
      ld4s(p.g_next, p.g_next_dtype, o, gn);
#pragma unroll
      for (int j = 0; j < 4; ++j) { gv[j] = fmaf(sn[j], gn[j], gv[j]); a_next[j] = fmaf(gn[j], v[j], a_next[j]); }
    }
    if (p.g_rgb) {
      const float4 gr = __ldg(reinterpret_cast<const float4*>(p.g_rgb + (n * HW + pix) * 4));
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 w = s_w[c + j];
        const float t = w.x * gr.x + w.y * gr.y + w.z * gr.z + w.w * gr.w;
        gv[j] = fmaf(sr[j], t, gv[j]);
        a_rgb[j] = fmaf(t, v[j], a_rgb[j]);
      }
    }
    if (p.g_y == nullptr) continue;
    float gy[4];
    const float nz = p.noise != nullptr ? p.noise_w * __ldg(p.noise + pix) : 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool pos = v[j] > 0.f;
      const float gp = gv[j] * (pos ? kpos : kneg);
      const float pre = v[j] * (pos ? 1.f / kpos : 1.f / kneg);
      a_dem[j] = fmaf(gp, pre - nz - bs[j], a_dem[j]);
      gy[j] = gp * dm[j];
    }
    int64_t dst = o;
    if (p.phases) {
      const int x = pix % p.W, yy = pix / p.W;
      const int ph = (yy & 1) * 2 + (x & 1);
      dst = (((n * (p.H >> 1) + (yy >> 1)) * (p.W >> 1) + (x >> 1)) * 4 + ph) * p.C + c;
    }
    st4s(p.g_y, p.g_y_dtype, dst, gy);
  }
  float* const accs[3] = {a_next, a_rgb, a_dem};
  float* const dsts[3] = {p.dot_next, p.dot_rgb, p.dot_demod};
  for (int k = 0; k < 3; ++k) {
    if (dsts[k] == nullptr) continue;                  // uniform across the block
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) red[threadIdx.x * 4 + j] = accs[k][j];
    __syncthreads();
    if (lane == 0) {
      float s[4] = {0.f, 0.f, 0.f, 0.f};
      for (int l = 0; l < lanes; ++l)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[j] += red[(l * c4n + cg) * 4 + j];
      float* d = dsts[k] + (n * p.parts + part) * p.C + c;
#pragma unroll
      for (int j = 0; j < 4; ++j) d[j] = s[j];
    }
  }
}

// ds[n][c] = sum_parts dot_mod[n][.][c] - s[n][c] * sum_o (sum_parts dot_demod[n][.][o]) * demod[n][o]^2 * wsq[o][c]
// (the modulation term and the demodulation adjoint d demod_o / d s_c = -demod_o^3 s_c wsq[o][c]); one block per sample.
__global__ void __launch_bounds__(256) style_bwd_kernel(const float* __restrict__ dot_mod, int parts_mod, const float* __restrict__ dot_demod,
                                                        int parts_demod, const float* __restrict__ s, const float* __restrict__ demod,
                                                        const float* __restrict__ wsq, int cin, int cout, float* __restrict__ ds) {
  extern __shared__ float q[];                          // [cout]
  const int64_t n = blockIdx.x;
  if (dot_demod != nullptr) {
    for (int o = threadIdx.x; o < cout; o += 256) {
      float a = 0.f;
      for (int pp = 0; pp < parts_demod; ++pp) a += dot_demod[(n * parts_demod + pp) * cout + o];
      const float d = demod[n * cout + o];
      q[o] = a * d * d;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < cin; c += 256) {
    float m = 0.f;
    if (dot_mod != nullptr)
      for (int pp = 0; pp < parts_mod; ++pp) m += dot_mod[(n * parts_mod + pp) * cin + c];
    if (dot_demod != nullptr) {
      float t = 0.f;
      for (int o = 0; o < cout; ++o) t = fmaf(q[o], __ldg(wsq + (int64_t)o * cin + c), t);
      m = fmaf(-s[n * cin + c], t, m);
    }
    ds[n * cin + c] = m;
  }
}

// adjoint of image_pool_out_kernel: g_o = g_purified * out_scale + g_cls, spread evenly over the k1 x k1 (x k2 x k2) source pixels;
// masked rows (set to -1 by the forward) pass no gradient.  One thread per generator pixel, float4 store (4th channel = padding, 0).
__global__ void image_pool_out_bwd_kernel(const float* __restrict__ g_pur, const void* g_cls, int cls_dtype, int N, int S, int k1, int k2,
                                          int mask_rows, float out_scale, float* __restrict__ g_img) {
  const int Sp = S / k1, So = Sp / k2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;        // over (n, Y, X)
  if (idx >= (int64_t)N * S * S) return;
  const int X = (int)(idx % S);
  const int Y = (int)((idx / S) % S);
  const int64_t n = idx / ((int64_t)S * S);
  const int r = Y / k1, q = X / k1;
  const int y = r / k2, x = q / k2;
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  if (!(r < mask_rows || r >= Sp - mask_rows)) {
    const float inv = 1.f / (float)(k1 * k1 * k2 * k2);
    for (int c = 0; c < 3; ++c) {
      float a = 0.f;
      if (g_pur != nullptr) a = g_pur[((n * 3 + c) * So + y) * So + x] * out_scale;
      if (g_cls != nullptr) a += ld1s(g_cls, cls_dtype, ((n * So + y) * So + x) * 3 + c);
      g[c] = a * inv;
    }
  }
  *reinterpret_cast<float4*>(g_img + idx * 4) = make_float4(g[0], g[1], g[2], g[3]);
}

// adjoint of latent_lerp w.r.t. the codes: g_codes[b,l,:] = (1 - a_l) * g_out[b,l,:]
__global__ void latent_lerp_bwd_kernel(const float* __restrict__ g_out, const float* __restrict__ alphas, int L, int D, int64_t total,
                                       float* __restrict__ g_codes) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  g_codes[i] = (1.f - alphas[(i / D) % L]) * g_out[i];
}

}  // namespace ga

using namespace ga;

extern "C" int ga_pixelnorm(const float* x, int rows, int d, const ga_tensor* out, void* stream) {
  GA_CHECK(x && out && rows >= 0 && d > 0 && numel(out) == (int64_t)rows * d, "ga_pixelnorm: bad arguments");
  if (rows == 0) return 0;
  pixelnorm_kernel<<<cdiv((int64_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(x, rows, d, out->data, out->dtype);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_style_demod(const float* s, const float* wsq, int n, int cin, int cout, float* demod, void* stream) {
  GA_CHECK(s && wsq && demod && n >= 0 && cin > 0 && cout > 0, "ga_style_demod: bad arguments");
  if (n == 0) return 0;
  style_demod_kernel<<<cdiv((int64_t)n * cout * 32, 256), 256, 0, (cudaStream_t)stream>>>(s, wsq, n, cin, cout, demod);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_channel_scale(const ga_tensor* x, const float* s, const ga_tensor* out, void* stream) {
  GA_CHECK(x && s && out && same_shape(x, out) && (x->c % 4) == 0, "ga_channel_scale: shape mismatch (channels must be a multiple of 4)");
  const int64_t total4 = numel(x) / 4;
  if (total4 == 0) return 0;
  channel_scale_kernel<<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(x->data, x->dtype, s, x->h * x->w, x->c, total4, out->data, out->dtype);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_styled_bias_act(const ga_tensor* y, int phases, const float* demod, const float* noise_hw, float noise_w,
                                  const float* bias, int act, const ga_tensor* skip, const float* skip_up_kernel, const float* scale_a,
                                  const ga_tensor* out, const float* scale_b, const ga_tensor* out_b, void* stream) {
  GA_CHECK(y && (out || out_b), "ga_styled_bias_act: null argument");
  const ga_tensor* o = out ? out : out_b;
  GA_CHECK((o->c % 4) == 0, "ga_styled_bias_act: channels must be a multiple of 4");
  if (phases) GA_CHECK(y->n == o->n && y->h * 2 == o->h && y->w * 2 == o->w && y->c == 4 * o->c, "ga_styled_bias_act: phase tensor must be [n][h/2][w/2][4*c]");
  else GA_CHECK(same_shape(y, o), "ga_styled_bias_act: shape mismatch");
  if (skip_up_kernel) GA_CHECK(skip && skip->n == o->n && skip->h * 2 == o->h && skip->w * 2 == o->w && skip->c == o->c,
                               "ga_styled_bias_act: an up-sampled skip must have half the output resolution");
  else GA_CHECK(!skip || same_shape(skip, o), "ga_styled_bias_act: skip shape mismatch");
  GA_CHECK(!out_b || (scale_b && (!out || same_shape(out, out_b))), "ga_styled_bias_act: out_b needs scale_b and out's shape");
  const int64_t total = numel(o) / 4;
  if (total == 0) return 0;
  {
    static int fast_on = -1;
    if (fast_on < 0) { const char* e = getenv("GA_SBA_FAST"); fast_on = e ? atoi(e) : 1; }
    const int lw = ilog2_exact(o->w), lh = ilog2_exact(o->h), lc8 = (o->c % 8 == 0) ? ilog2_exact(o->c / 8) : -1;
    const bool bf_out = (!out || out->dtype == GA_BF16) && (!out_b || out_b->dtype == GA_BF16);
    if (fast_on && !skip && act == GA_ACT_LRELU_SQRT2 && bf_out && lw >= 1 && lh >= 1 && lc8 >= 0 && numel(o) / 8 < (int64_t)0x7fffff00 &&
        (int64_t)o->n * o->c < (int64_t)0x7fffffff && (((uintptr_t)y->data) & 15) == 0 && (!out || (((uintptr_t)out->data) & 15) == 0) &&
        (!out_b || (((uintptr_t)out_b->data) & 15) == 0)) {
      SbaFast p;
      p.y = y->data; p.demod = demod; p.noise = noise_hw; p.bias = bias; p.scale_a = scale_a; p.scale_b = scale_b;
      p.out = out ? (__nv_bfloat16*)out->data : nullptr; p.out_b = out_b ? (__nv_bfloat16*)out_b->data : nullptr;
      p.noise_w = noise_w; p.lw = lw; p.lh = lh; p.lc8 = lc8; p.total = (uint32_t)(numel(o) / 8);
      const unsigned grid = (unsigned)cdiv((int64_t)p.total, 256 * 4);
      cudaStream_t st = (cudaStream_t)stream;
      if (phases) {
        if (y->dtype == GA_F32) styled_bias_act_vec8_kernel<true, true><<<grid, 256, 0, st>>>(p);
        else styled_bias_act_vec8_kernel<true, false><<<grid, 256, 0, st>>>(p);
      } else {
        if (y->dtype == GA_F32) styled_bias_act_vec8_kernel<false, true><<<grid, 256, 0, st>>>(p);
        else styled_bias_act_vec8_kernel<false, false><<<grid, 256, 0, st>>>(p);
      }
      GA_LAUNCH_OK();
      return 0;
    }
  }
  styled_bias_act_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(y->data, y->dtype, phases, demod, noise_hw, noise_w, bias, act,
                                                                              skip ? skip->data : nullptr, skip ? skip->dtype : GA_F32, o->n,
                                                                              o->h, o->w, o->c, scale_a, out ? out->data : nullptr,
                                                                              out ? out->dtype : GA_F32, scale_b, out_b ? out_b->data : nullptr,
                                                                              out_b ? out_b->dtype : GA_F32, skip_up_kernel);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_torgb_fused(const ga_tensor* x, const void* w_bf16, const float* bias, const ga_tensor* skip, const float* skip_up_kernel,
                              const ga_tensor* out, void* stream) {
  GA_CHECK(x && w_bf16 && out, "ga_torgb_fused: null argument");
  GA_CHECK(x->dtype == GA_BF16 && (x->c % 8) == 0 && out->dtype == GA_F32 && out->c == 4 && out->n == x->n && out->h == x->h && out->w == x->w,
           "ga_torgb_fused: x must be bf16 with channels %% 8 == 0, out fp32 [n][h][w][4]");
  GA_CHECK((skip == nullptr) == (skip_up_kernel == nullptr), "ga_torgb_fused: skip and its up-sampling kernel go together");
  if (skip) GA_CHECK(skip->dtype == GA_F32 && skip->c == 4 && skip->n == x->n && skip->h * 2 == x->h && skip->w * 2 == x->w,
                     "ga_torgb_fused: skip must be fp32 [n][h/2][w/2][4]");
  GA_CHECK(((((uintptr_t)x->data) | ((uintptr_t)out->data) | (skip ? (uintptr_t)skip->data : 0) | (bias ? (uintptr_t)bias : 0)) & 15) == 0,
           "ga_torgb_fused: pointers must be 16-byte aligned");
  const int64_t pixels = (int64_t)x->n * x->h * x->w;
  if (pixels == 0) return 0;
  const size_t smem = (size_t)x->c * sizeof(float4);
  GA_CHECK(smem <= 48 * 1024, "ga_torgb_fused: too many input channels");
  torgb_fused_kernel<<<(unsigned)cdiv(pixels, 256), 256, smem, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)x->data, (const __nv_bfloat16*)w_bf16, bias, skip ? (const float*)skip->data : nullptr, skip_up_kernel, x->n, x->h, x->w,
      x->c, (float*)out->data);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_upfirdn2d(const ga_tensor* in, const float* kernel, int kh, int kw, int up, int down, int pad0, int pad1,
                            const ga_tensor* out, void* stream) {
  GA_CHECK(in && kernel && out && up >= 1 && down >= 1 && kh >= 1 && kw >= 1, "ga_upfirdn2d: bad arguments");
  const int Ho = (in->h * up + pad0 + pad1 - kh) / down + 1, Wo = (in->w * up + pad0 + pad1 - kw) / down + 1;
  GA_CHECK(out->n == in->n && out->c == in->c && out->h == Ho && out->w == Wo, "ga_upfirdn2d: output must be (%d,%d,%d,%d)", in->n, Ho, Wo, in->c);
  const int64_t total = numel(out);
  if (total == 0) return 0;
  upfirdn2d_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, kernel, kh, kw, up, down, pad0, in->n, in->h, in->w,
                                                                       in->c, Ho, Wo, out->data, out->dtype);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_avgpool_to_nchw(const ga_tensor* in, int k, int out_c, float* out_nchw, void* stream) {
  GA_CHECK(in && out_nchw && k >= 1 && in->h % k == 0 && in->w % k == 0 && out_c >= 1 && out_c <= in->c, "ga_avgpool_to_nchw: bad arguments");
  const int64_t total = (int64_t)in->n * out_c * (in->h / k) * (in->w / k);
  if (total == 0) return 0;
  avgpool_to_nchw_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, in->n, in->h, in->w, in->c, out_c, k, out_nchw);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_latent_lerp(const float* codes, const float* styles, const float* alphas_dev, int b, int l, int d, float* out, void* stream) {
  GA_CHECK(codes && styles && alphas_dev && out && b >= 0 && l > 0 && d > 0, "ga_latent_lerp: bad arguments");
  const int64_t total = (int64_t)b * l * d;
  if (total == 0) return 0;
  latent_lerp_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(codes, styles, alphas_dev, l, d, total, out);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_styled_bias_act_bwd_parts(int hw, int c) {
  if (hw <= 0 || c <= 0) return 0;
  const int ppp = sba_bwd_pix_per_part(c);
  return (hw + ppp - 1) / ppp;
}

extern "C" int ga_styled_bias_act_bwd(const ga_tensor* v, const ga_tensor* g_next, const float* s_next, const float* g_rgb, const float* w_rgb,
                                      const float* s_rgb, const float* demod, const float* noise_hw, float noise_w, const float* bias, int phases,
                                      const ga_tensor* g_y, float* dot_next, float* dot_rgb, float* dot_demod, void* stream) {
  GA_CHECK(v && (g_next || g_rgb), "ga_styled_bias_act_bwd: null argument");
  const int C = v->c;
  GA_CHECK(C % 4 == 0 && C / 4 <= 256 && 256 % (C / 4) == 0, "ga_styled_bias_act_bwd: channels must be 4 * a power of two <= 1024, got %d", C);
  GA_CHECK(!g_next || same_shape(g_next, v), "ga_styled_bias_act_bwd: g_next must have the activation's shape");
  GA_CHECK(!g_rgb || (w_rgb && s_rgb), "ga_styled_bias_act_bwd: the RGB branch needs its weights and style");
  GA_CHECK(!dot_rgb || g_rgb, "ga_styled_bias_act_bwd: dot_rgb needs g_rgb");
  GA_CHECK(!g_y || demod, "ga_styled_bias_act_bwd: g_y needs demod");
  GA_CHECK(!dot_demod || g_y, "ga_styled_bias_act_bwd: dot_demod needs g_y");
  if (g_y) {
    if (phases) GA_CHECK(v->h % 2 == 0 && v->w % 2 == 0 && g_y->n == v->n && g_y->h * 2 == v->h && g_y->w * 2 == v->w && g_y->c == 4 * C,
                         "ga_styled_bias_act_bwd: phase gradient must be [n][h/2][w/2][4*c]");
    else GA_CHECK(same_shape(g_y, v), "ga_styled_bias_act_bwd: g_y shape mismatch");
  }
  // 4-channel vectors: 16 bytes in fp32, 8 in bf16
  auto vec_aligned = [](const ga_tensor* t) { return !t || (((uintptr_t)t->data) % (t->dtype == GA_F32 ? 16 : 8)) == 0; };
  GA_CHECK(vec_aligned(v) && vec_aligned(g_next) && vec_aligned(g_y) && (((uintptr_t)g_rgb) | ((uintptr_t)w_rgb)) % 16 == 0,
           "ga_styled_bias_act_bwd: tensors must be aligned to 4 channels (g_rgb / w_rgb to 16 bytes)");
  const int hw = v->h * v->w;
  if ((int64_t)v->n * hw == 0) return 0;
  GA_CHECK(v->n <= 65535, "ga_styled_bias_act_bwd: batch too large");
  SbaBwd p;
  p.v = v->data; p.v_dtype = v->dtype;
  p.g_next = g_next ? g_next->data : nullptr; p.g_next_dtype = g_next ? g_next->dtype : GA_F32; p.s_next = s_next;
  p.g_rgb = g_rgb; p.w_rgb = g_rgb ? w_rgb : nullptr; p.s_rgb = s_rgb;
  p.demod = demod; p.noise = noise_hw; p.noise_w = noise_w; p.bias = bias;
  p.g_y = g_y ? g_y->data : nullptr; p.g_y_dtype = g_y ? g_y->dtype : GA_F32; p.phases = phases;
  p.dot_next = g_next ? dot_next : nullptr; p.dot_rgb = dot_rgb; p.dot_demod = dot_demod;
  p.H = v->h; p.W = v->w; p.C = C; p.ppp = sba_bwd_pix_per_part(C); p.parts = ga_styled_bias_act_bwd_parts(hw, C);
  const size_t smem = (size_t)(p.w_rgb ? C * 4 : 0) * sizeof(float) + 256 * 4 * sizeof(float);
  GA_CHECK(smem <= 48 * 1024, "ga_styled_bias_act_bwd: too many channels");
  styled_bias_act_bwd_kernel<<<dim3(p.parts, v->n), 256, smem, (cudaStream_t)stream>>>(p);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_style_bwd(const float* dot_mod, int parts_mod, const float* dot_demod, int parts_demod, const float* s, const float* demod,
                            const float* wsq, int n, int cin, int cout, float* ds, void* stream) {
  GA_CHECK(ds && n >= 0 && cin > 0 && (dot_mod || dot_demod), "ga_style_bwd: bad arguments");
  GA_CHECK(!dot_mod || parts_mod > 0, "ga_style_bwd: parts_mod must be positive");
  GA_CHECK(!dot_demod || (parts_demod > 0 && s && demod && wsq && cout > 0), "ga_style_bwd: the demodulation term needs s, demod, wsq, cout");
  if (n == 0) return 0;
  const size_t smem = dot_demod ? (size_t)cout * sizeof(float) : 0;
  GA_CHECK(smem <= 48 * 1024, "ga_style_bwd: too many output channels");
  style_bwd_kernel<<<n, 256, smem, (cudaStream_t)stream>>>(dot_mod, parts_mod, dot_demod, parts_demod, s, demod, wsq, cin, cout, ds);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_image_pool_out_bwd(const float* g_purified_nchw, const ga_tensor* g_cls, int k1, int k2, int mask_rows, float out_scale,
                                     const ga_tensor* g_img, void* stream) {
  GA_CHECK(g_img && g_img->dtype == GA_F32 && g_img->c == 4 && g_img->h == g_img->w && k1 >= 1 && (k2 == 1 || k2 == 2) &&
               g_img->h % (k1 * k2) == 0 && mask_rows >= 0 && (g_purified_nchw || g_cls),
           "ga_image_pool_out_bwd: bad arguments");
  const int so = g_img->h / (k1 * k2);
  GA_CHECK(!g_cls || (g_cls->n == g_img->n && g_cls->h == so && g_cls->w == so && g_cls->c == 3), "ga_image_pool_out_bwd: g_cls shape mismatch");
  GA_CHECK((((uintptr_t)g_img->data) & 15) == 0, "ga_image_pool_out_bwd: g_img must be 16-byte aligned");
  const int64_t total = numel(g_img) / 4;
  if (total == 0) return 0;
  image_pool_out_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(g_purified_nchw, g_cls ? g_cls->data : nullptr,
                                                                                g_cls ? g_cls->dtype : GA_F32, g_img->n, g_img->h, k1, k2,
                                                                                mask_rows, out_scale, (float*)g_img->data);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_latent_lerp_bwd(const float* g_out, const float* alphas_dev, int b, int l, int d, float* g_codes, void* stream) {
  GA_CHECK(g_out && alphas_dev && g_codes && b >= 0 && l > 0 && d > 0, "ga_latent_lerp_bwd: bad arguments");
  const int64_t total = (int64_t)b * l * d;
  if (total == 0) return 0;
  latent_lerp_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(g_out, alphas_dev, l, d, total, g_codes);
  GA_LAUNCH_OK();
  return 0;
}
