// Input-gradient (dgrad-only) kernels of the purification path: the attack path of the reference runs
// `torch.autograd.grad(loss, [x])` through classifier -> decoder -> latent mix -> encoder -> noise/blur
// (/root/reference/src/attacks/untargeted.py:146,201).  All weights are frozen, so no weight gradient exists
// anywhere here (the reference computes them and throws them away, SURVEY Appendix F).
// Convolution dgrads re-use the forward conv kernels on flipped/transposed weights; this file holds the
// bandwidth-bound pieces.  Reductions are two-stage without atomics (bit-reproducible).
#include <stdlib.h>
#include "ga_common.cuh"

namespace ga {

__device__ __forceinline__ float ld1b(const void* base, int dtype, int64_t off) {
  return dtype == GA_F32 ? reinterpret_cast<const float*>(base)[off]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[off]);
}
__device__ __forceinline__ void st1b(void* base, int dtype, int64_t off, float v) {
  if (dtype == GA_F32) reinterpret_cast<float*>(base)[off] = v;
  else reinterpret_cast<__nv_bfloat16*>(base)[off] = __float2bfloat16_rn(v);
}
__device__ __forceinline__ float sc5_grad(float t) {   // d/dt 5 tanh(t/5)
  const float th = tanhf(t * 0.2f);
  return 1.0f - th * th;
}

// ---------------------------------------------------------------------------- pre-activation backward
// out = g * act'(scale*x + shift) * scale (+ add)
__global__ void affine_act_bwd_kernel(const void* g, int g_dtype, const void* x, int x_dtype, const float* __restrict__ scale,
                                      const float* __restrict__ shift, int act, const void* add, int add_dtype, void* out,
                                      int out_dtype, int C, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  float sc = 1.f, sh = 0.f;
  if (scale != nullptr) { sc = scale[c]; sh = shift[c]; }
  float v = ld1b(g, g_dtype, i) * act_grad(fmaf(ld1b(x, x_dtype, i), sc, sh), act) * sc;
  if (add != nullptr) v += ld1b(add, add_dtype, i);
  st1b(out, out_dtype, i, v);
}

__global__ void __launch_bounds__(256) affine_act_bwd_vec4_kernel(const void* g, int g_dtype, const void* x, int x_dtype,
                                                                  const float* __restrict__ scale, const float* __restrict__ shift, int act,
                                                                  const void* add, int add_dtype, void* out, int out_dtype, int C,
                                                                  int64_t total4) {
  int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const int64_t i = i4 * 4;
  const int c = (int)(i % C);
  float gv[4], xv[4], av[4] = {0.f, 0.f, 0.f, 0.f}, o[4];
  if (g_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(g) + i, gv); else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(g) + i, gv);
  if (x_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(x) + i, xv); else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(x) + i, xv);
  if (add != nullptr) {
    if (add_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(add) + i, av); else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(add) + i, av);
  }
  float sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
  if (scale != nullptr) {
    const float4 s4 = __ldg(reinterpret_cast<const float4*>(scale + c)), h4 = __ldg(reinterpret_cast<const float4*>(shift + c));
    sc[0] = s4.x; sc[1] = s4.y; sc[2] = s4.z; sc[3] = s4.w; sh[0] = h4.x; sh[1] = h4.y; sh[2] = h4.z; sh[3] = h4.w;
  }
  float pre4[4], d4[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) pre4[j] = fmaf(xv[j], sc[j], sh[j]);
  act_grad_n<4>(pre4, d4, act);
#pragma unroll
  for (int j = 0; j < 4; ++j) o[j] = fmaf(gv[j] * d4[j], sc[j], av[j]);
  if (out_dtype == GA_F32) st4<float>(reinterpret_cast<float*>(out) + i, o); else st4<__nv_bfloat16>(reinterpret_cast<__nv_bfloat16*>(out) + i, o);
}

// out = a + b  (gradient accumulation)
__global__ void add_kernel(const void* a, int a_dtype, const void* b, int b_dtype, void* out, int out_dtype, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  st1b(out, out_dtype, i, ld1b(a, a_dtype, i) + ld1b(b, b_dtype, i));
}

// fp32 + fp32 -> fp32 with 16-byte vectors, 4 per thread (the gradient accumulations of the attack path: stash / skip joins)
__global__ void __launch_bounds__(256) add_f32x4_kernel(const float4* __restrict__ a, const float4* __restrict__ b, float4* __restrict__ out, int64_t total4) {
  const int64_t i0 = (int64_t)blockIdx.x * 1024 + threadIdx.x;
  float4 va[4], vb[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t i = i0 + u * 256;
    if (i < total4) { va[u] = __ldg(a + i); vb[u] = __ldg(b + i); }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t i = i0 + u * 256;
    if (i < total4) out[i] = make_float4(va[u].x + vb[u].x, va[u].y + vb[u].y, va[u].z + vb[u].z, va[u].w + vb[u].w);
  }
}

// ---------------------------------------------------------------------------- SE + residual backward
// forward: out = skip + s * gate[n,c] * r ;  gate = sigmoid(W2 relu(W1 mean(r) + b1) + b2)   (b1 / b2 may be null: no bias)
// stage 1: dots[n][blk][c] = sum over the block's pixel slice of g_out * r
__global__ void __launch_bounds__(256) se_bwd_reduce_kernel(const void* __restrict__ g, int g_dtype, const void* __restrict__ r,
                                                            int r_dtype, int HW, int C, int pix_per_block,
                                                            float* __restrict__ partial) {
  __shared__ float s_part[256];
  const int n = blockIdx.y;
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(p0 + pix_per_block, HW);
  const int64_t base = ((int64_t)n * HW + p0) * C;
  const int cnt = (p1 - p0) * C;
  float* dst = partial + ((int64_t)n * gridDim.x + blockIdx.x) * C;
  const int cg = C >> 2;                       // 4-channel groups
  if ((C & 3) == 0 && cg <= 256 && 256 % cg == 0) {
    // vector path: a thread owns 4 channels of every PL-th pixel (16-byte fp32 / 8-byte bf16 loads, 4 pixels in flight per thread);
    // the pixel lanes are then added in fixed order (bit-reproducible)
    __shared__ float s_vec[256][4];
    const int PL = 256 / cg;
    const int g4 = threadIdx.x % cg, pl = threadIdx.x / cg;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const int npix = p1 - p0;
    for (int q0 = pl; q0 < npix; q0 += 4 * PL) {
      float gv[4][4], rv[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int q = q0 + u * PL;
        if (q < npix) {
          const int64_t off = base + (int64_t)q * C + 4 * g4;
          if (g_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(g) + off, gv[u]);
          else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(g) + off, gv[u]);
          if (r_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(r) + off, rv[u]);
          else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(r) + off, rv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (q0 + u * PL < npix) {
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[j] = fmaf(gv[u][j], rv[u][j], acc[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) s_vec[threadIdx.x][j] = acc[j];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
      float t = 0.f;
      for (int l = 0; l < PL; ++l) t += s_vec[l * cg + (c >> 2)][c & 3];
      dst[c] = t;
    }
  } else if (256 % C == 0) {
    float acc = 0.f;
    for (int i = threadIdx.x; i < cnt; i += 256) acc = fmaf(ld1b(g, g_dtype, base + i), ld1b(r, r_dtype, base + i), acc);
    s_part[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < C) {
      float t = 0.f;
      for (int k = threadIdx.x; k < 256; k += C) t += s_part[k];
      dst[threadIdx.x] = t;
    }
  } else if (C % 256 == 0) {
    for (int k = 0; k < C / 256; ++k) {
      float acc = 0.f;
      for (int i = threadIdx.x + k * 256; i < cnt; i += C) acc = fmaf(ld1b(g, g_dtype, base + i), ld1b(r, r_dtype, base + i), acc);
      dst[threadIdx.x + k * 256] = acc;
    }
  } else {
    for (int c = threadIdx.x; c < C; c += 256) {
      float acc = 0.f;
      for (int i = c; i < cnt; i += C) acc = fmaf(ld1b(g, g_dtype, base + i), ld1b(r, r_dtype, base + i), acc);
      dst[c] = acc;
    }
  }
}

struct SeBwdParams {
  const void* g; int g_dtype;
  const float* sums; const float* dots;
  const float* w1; const float* b1; const float* w2; const float* b2;
  int hidden; float res_scale;
  void* g_r; int gr_dtype;
  int HW, C, pix_per_block, nparts;
};

// stage 2: g_r = s * gate * g_out + g_mean / HW, with g_mean from the 2-layer gate MLP backward (recomputed per CTA)
__global__ void __launch_bounds__(256) se_bwd_apply_kernel(SeBwdParams p) {
  extern __shared__ float sm[];    // mean[C] | gate[C] | gmean[C] | hid[h] | ghid[h] | ga2[C]
  float* s_mean = sm;
  float* s_gate = sm + p.C;
  float* s_gmean = sm + 2 * p.C;
  float* s_ga2 = sm + 3 * p.C;
  float* s_hid = sm + 4 * p.C;
  float* s_ghid = s_hid + p.hidden;
  const int n = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float inv = 1.0f / (float)p.HW;
  for (int c = tid; c < p.C; c += 256) {
    float t = 0.f, d = 0.f;
    for (int k = 0; k < p.nparts; ++k) {
      t += p.sums[((int64_t)n * p.nparts + k) * p.C + c];
      d += p.dots[((int64_t)n * p.nparts + k) * p.C + c];
    }
    s_mean[c] = t * inv;
    s_gmean[c] = d;                // temporarily: sum_p g_out * r
  }
  __syncthreads();
  for (int j = warp; j < p.hidden; j += 8) {
    float a = 0.f;
    for (int c = lane; c < p.C; c += 32) a = fmaf(p.w1[(int64_t)j * p.C + c], s_mean[c], a);
    a = warp_sum(a);
    if (lane == 0) s_hid[j] = a + (p.b1 != nullptr ? p.b1[j] : 0.f);          // pre-ReLU
  }
  __syncthreads();
  for (int c = tid; c < p.C; c += 256) {
    float a = p.b2 != nullptr ? p.b2[c] : 0.f;
    for (int j = 0; j < p.hidden; ++j) a = fmaf(p.w2[(int64_t)c * p.hidden + j], fmaxf(s_hid[j], 0.f), a);
    const float gt = sigmoidf_(a);
    s_gate[c] = gt;
    s_ga2[c] = p.res_scale * s_gmean[c] * gt * (1.f - gt);     // d loss / d (pre-sigmoid)
  }
  __syncthreads();
  for (int j = warp; j < p.hidden; j += 8) {
    float a = 0.f;
    for (int c = lane; c < p.C; c += 32) a = fmaf(p.w2[(int64_t)c * p.hidden + j], s_ga2[c], a);
    a = warp_sum(a);
    if (lane == 0) s_ghid[j] = s_hid[j] > 0.f ? a : 0.f;
  }
  __syncthreads();
  for (int c = tid; c < p.C; c += 256) {
    float a = 0.f;
    for (int j = 0; j < p.hidden; ++j) a = fmaf(p.w1[(int64_t)j * p.C + c], s_ghid[j], a);
    s_gmean[c] = a * inv;                             // d loss / d r through the mean, per pixel
  }
  __syncthreads();
  const int p0 = blockIdx.x * p.pix_per_block;
  const int p1 = min(p0 + p.pix_per_block, p.HW);
  const int64_t base = ((int64_t)n * p.HW + p0) * p.C;
  const int cnt = (p1 - p0) * p.C;
  if ((p.C & 3) == 0) {
    const int c4n = p.C >> 2, cnt4 = cnt >> 2;
    for (int i0 = tid; i0 < cnt4; i0 += 256 * 4) {       // 4 vectors per thread in flight
      float gv[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * 256;
        if (i < cnt4) {
          if (p.g_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(p.g) + base + (int64_t)i * 4, gv[u]);
          else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(p.g) + base + (int64_t)i * 4, gv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * 256;
        if (i >= cnt4) continue;
        const int c = (i % c4n) * 4;
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = fmaf(p.res_scale * s_gate[c + j], gv[u][j], s_gmean[c + j]);
        if (p.gr_dtype == GA_F32) st4<float>(reinterpret_cast<float*>(p.g_r) + base + (int64_t)i * 4, o);
        else st4<__nv_bfloat16>(reinterpret_cast<__nv_bfloat16*>(p.g_r) + base + (int64_t)i * 4, o);
      }
    }
    return;
  }
  for (int i = tid; i < cnt; i += 256) {
    const int c = i % p.C;
    st1b(p.g_r, p.gr_dtype, base + i, fmaf(p.res_scale * s_gate[c], ld1b(p.g, p.g_dtype, base + i), s_gmean[c]));
  }
}

// ---------------------------------------------------------------------------- resampling backward
__global__ void sumpool2x2_kernel(const void* in, int in_dtype, const void* mul, int mul_dtype, void* out, int out_dtype, int N, int Ho,
                                  int Wo, int C) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * C) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  const int W = 2 * Wo;
  const int64_t b = ((n * 2 * Ho + 2 * y) * W + 2 * x) * C + c;
  float v = ld1b(in, in_dtype, b) + ld1b(in, in_dtype, b + C) + ld1b(in, in_dtype, b + (int64_t)W * C) +
            ld1b(in, in_dtype, b + (int64_t)W * C + C);
  if (mul != nullptr) v *= ld1b(mul, mul_dtype, idx);
  st1b(out, out_dtype, idx, v);
}

// 4 channels per thread (C % 4 == 0): 16-byte fp32 / 8-byte bf16 accesses
__global__ void __launch_bounds__(256) sumpool2x2_vec4_kernel(const void* __restrict__ in, int in_dtype, const void* __restrict__ mul,
                                                              int mul_dtype, void* __restrict__ out, int out_dtype, int64_t total4, int Ho,
                                                              int Wo, int C) {
  const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const int c4n = C >> 2;
  const int c = (int)(i4 % c4n) * 4;
  int64_t t = i4 / c4n;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  const int W = 2 * Wo;
  const int64_t b = ((n * 2 * Ho + 2 * y) * W + 2 * x) * C + c;
  float a0[4], a1[4], a2[4], a3[4], o[4];
  auto ld = [&](const void* base, int dt, int64_t off, float (&v)[4]) {
    if (dt == GA_F32) ld4<float>(reinterpret_cast<const float*>(base) + off, v);
    else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(base) + off, v);
  };
  ld(in, in_dtype, b, a0); ld(in, in_dtype, b + C, a1); ld(in, in_dtype, b + (int64_t)W * C, a2); ld(in, in_dtype, b + (int64_t)W * C + C, a3);
#pragma unroll
  for (int j = 0; j < 4; ++j) o[j] = (a0[j] + a1[j]) + (a2[j] + a3[j]);
  const int64_t oi = i4 * 4;
  if (mul != nullptr) {
    float m[4];
    ld(mul, mul_dtype, oi, m);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] *= m[j];
  }
  if (out_dtype == GA_F32) st4<float>(reinterpret_cast<float*>(out) + oi, o);
  else st4<__nv_bfloat16>(reinterpret_cast<__nv_bfloat16*>(out) + oi, o);
}

// depth-to-space x2: out[n][2a+pi][2b+pj][c] = in[n][a][b][(2 pi + pj) C + c].  The input gradient of a stride-2 convolution is computed
// as ONE stride-1 tensor-core conv over grad_out that emits the four output phases as 4C channels (nvae_engine._build_dgrad); this kernel
// interleaves them.  4 channels per thread: reads and writes are 16-byte vectors on contiguous channel runs.
__global__ void __launch_bounds__(256) depth_to_space2_kernel(const float4* __restrict__ in, float4* __restrict__ out, int64_t total4, int h,
                                                              int w, int c4) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // over the OUTPUT, channel-vector granularity
  if (idx >= total4) return;
  const int c = (int)(idx % c4);
  int64_t t = idx / c4;
  const int X = (int)(t % (2 * w)); t /= 2 * w;
  const int Y = (int)(t % (2 * h));
  const int64_t n = t / (2 * h);
  const int ph = (Y & 1) * 2 + (X & 1);
  out[idx] = __ldg(in + (((n * h + (Y >> 1)) * w + (X >> 1)) * 4 + ph) * c4 + c);
}

// depth_to_space2 with the rest of the dgrad epilogue: out = (d2s(in) + add) * f(mul), fp32 in, fp32 / bf16 out.  One pass over the four
// phases of a stride-2 conv's input gradient instead of d2s, add and mask as three; same arithmetic, in the same order, as those three.
template <typename TOut>
__global__ void __launch_bounds__(256) phase_interleave_kernel(const float4* __restrict__ in, const void* add, int add_dtype, const void* mul,
                                                               int mul_dtype, int mul_mode, const float* __restrict__ slope, TOut* __restrict__ out,
                                                               int64_t total4, int h, int w, int c4) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // over the OUTPUT, 4-channel vectors
  if (idx >= total4) return;
  const int c = (int)(idx % c4);
  int64_t t = idx / c4;
  const int X = (int)(t % (2 * w)); t /= 2 * w;
  const int Y = (int)(t % (2 * h));
  const int64_t n = t / (2 * h);
  const int ph = (Y & 1) * 2 + (X & 1);
  const float4 v4 = __ldg(in + (((n * h + (Y >> 1)) * w + (X >> 1)) * 4 + ph) * c4 + c);
  float v[4] = {v4.x, v4.y, v4.z, v4.w};
  const int64_t i = idx * 4;
  if (add != nullptr) {
    float a[4];
    if (add_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(add) + i, a); else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(add) + i, a);
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] += a[j];
  }
  if (mul != nullptr) {
    float m[4];
    if (mul_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(mul) + i, m); else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(mul) + i, m);
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] *= mul_factor(m[j], mul_mode, slope != nullptr ? __ldg(slope + 4 * c + j) : 0.f);
  }
  st4<TOut>(out + i, v);
}

// adjoint of the stride-2 sub-sample (MaxPool2d(1, 2)): every output pixel is written, the odd ones with zeros
__global__ void __launch_bounds__(256) subsample2x_bwd_kernel(const void* g, int g_dtype, void* out, int out_dtype, int64_t total4, int H, int W,
                                                              int c4, int Hg, int Wg) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total4) return;
  const int c = (int)(idx % c4);
  int64_t t = idx / c4;
  const int x = (int)(t % W); t /= W;
  const int y = (int)(t % H);
  const int64_t n = t / H;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (((x | y) & 1) == 0) {
    const int64_t gi = ((n * Hg + (y >> 1)) * Wg + (x >> 1)) * (4 * c4) + 4 * c;
    if (g_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(g) + gi, v); else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(g) + gi, v);
  }
  if (out_dtype == GA_F32) st4<float>(reinterpret_cast<float*>(out) + idx * 4, v); else st4<__nv_bfloat16>(reinterpret_cast<__nv_bfloat16*>(out) + idx * 4, v);
}

// transpose of the align_corners=True bilinear x2 up-sampling, as a deterministic gather
__global__ void bilinear2x_bwd_kernel(const void* g, int g_dtype, void* out, int out_dtype, int N, int H, int W, int C) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * H * W * C) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int x = (int)(t % W); t /= W;
  const int y = (int)(t % H);
  const int64_t n = t / H;
  const int Ho = 2 * H, Wo = 2 * W;
  const float sy = Ho > 1 ? (float)(H - 1) / (float)(Ho - 1) : 0.f;
  const float sx = Wo > 1 ? (float)(W - 1) / (float)(Wo - 1) : 0.f;
  // output rows whose source interval touches y: src = sy*oy in (y-1, y+1)
  const int oy_lo = sy > 0.f ? max(0, (int)floorf((y - 1) / sy)) : 0, oy_hi = sy > 0.f ? min(Ho - 1, (int)ceilf((y + 1) / sy)) : Ho - 1;
  const int ox_lo = sx > 0.f ? max(0, (int)floorf((x - 1) / sx)) : 0, ox_hi = sx > 0.f ? min(Wo - 1, (int)ceilf((x + 1) / sx)) : Wo - 1;
  float acc = 0.f;
  for (int oy = oy_lo; oy <= oy_hi; ++oy) {
    const float fy = sy * oy;
    int y0 = min((int)fy, H - 1);
    const int y1 = min(y0 + 1, H - 1);
    const float wy1 = fy - y0;
    float wy = 0.f;
    if (y0 == y) wy += 1.f - wy1;
    if (y1 == y) wy += wy1;
    if (wy == 0.f) continue;
    for (int ox = ox_lo; ox <= ox_hi; ++ox) {
      const float fx = sx * ox;
      int x0 = min((int)fx, W - 1);
      const int x1 = min(x0 + 1, W - 1);
      const float wx1 = fx - x0;
      float wx = 0.f;
      if (x0 == x) wx += 1.f - wx1;
      if (x1 == x) wx += wx1;
      if (wx == 0.f) continue;
      acc = fmaf(wy * wx, ld1b(g, g_dtype, ((n * Ho + oy) * Wo + ox) * C + c), acc);
    }
  }
  st1b(out, out_dtype, idx, acc);
}

// max-pool 2x2 backward: gradient goes to the FIRST maximal element of the window (torch semantics)
__global__ void maxpool2x2_bwd_kernel(const void* xin, int x_dtype, const void* g, int g_dtype, int relu, void* out, int out_dtype,
                                      int N, int H, int W, int C) {
  const int Ho = H >> 1, Wo = W >> 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // over pooled outputs
  if (idx >= (int64_t)N * Ho * Wo * C) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  const int64_t b = ((n * H + 2 * y) * W + 2 * x) * C + c;
  const int64_t o[4] = {b, b + C, b + (int64_t)W * C, b + (int64_t)W * C + C};
  float v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = ld1b(xin, x_dtype, o[k]);
  int best = 0;
#pragma unroll
  for (int k = 1; k < 4; ++k)
    if (v[k] > v[best]) best = k;
  float gv = ld1b(g, g_dtype, idx);
  if (relu && !(v[best] > 0.f)) gv = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) st1b(out, out_dtype, o[k], k == best ? gv : 0.f);
}


// max-pool 3x3 / stride 2 / pad 1 backward (torchvision ResNet stem), gather form without atomics: an input pixel belongs to up to four
// windows; it receives a window's gradient iff it is that window's FIRST maximum in scan order (torch's max_pool2d_with_indices backward).
// relu != 0: the pooled tensor is ReLU(conv): the gradient also passes the ReLU mask of the input value (stem conv -> ReLU -> pool).
__global__ void maxpool3x3s2_bwd_kernel(const void* xin, int x_dtype, const void* g, int g_dtype, int relu, void* out, int out_dtype,
                                        int N, int H, int W, int C) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // over input elements
  if (idx >= (int64_t)N * H * W * C) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int x = (int)(t % W); t /= W;
  const int y = (int)(t % H);
  const int64_t n = t / H;
  const float v = ld1b(xin, x_dtype, idx);
  float acc = 0.f;
  if (!(relu && !(v > 0.f))) {
    // windows (oy, ox) with 2*oy - 1 <= y <= 2*oy + 1
    for (int oy = (y) / 2; oy <= (y + 1) / 2; ++oy) {
      if (oy < 0 || oy >= Ho) continue;
      for (int ox = (x) / 2; ox <= (x + 1) / 2; ++ox) {
        if (ox < 0 || ox >= Wo) continue;
        // is (y, x) the first maximum of window (oy, ox)?
        bool first = true;
        for (int dy = -1; dy <= 1 && first; ++dy) {
          const int iy = 2 * oy + dy;
          if (iy < 0 || iy >= H) continue;
          for (int dx = -1; dx <= 1; ++dx) {
            const int ix = 2 * ox + dx;
            if (ix < 0 || ix >= W) continue;
            if (iy == y && ix == x) continue;
            const float u = ld1b(xin, x_dtype, ((n * H + iy) * W + ix) * C + c);
            const bool before = (iy < y) || (iy == y && ix < x);
            if (u > v || (before && u == v)) { first = false; break; }
          }
        }
        if (first) acc += ld1b(g, g_dtype, ((n * Ho + oy) * Wo + ox) * C + c);
      }
    }
  }
  st1b(out, out_dtype, idx, acc);
}

// global average pool backward fused with the ReLU mask of the pooled tensor: out[n,h,w,c] = g[n,c] / HW * (y[n,h,w,c] > 0)
__global__ void avgpool_bwd_relu_kernel(const void* g, int g_dtype, const void* y, int y_dtype, void* out, int out_dtype, int HW, int C,
                                        int64_t total) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = (int)(idx % C);
  const int64_t n = idx / ((int64_t)HW * C);
  const float m = ld1b(y, y_dtype, idx) > 0.f ? 1.f / (float)HW : 0.f;
  st1b(out, out_dtype, idx, ld1b(g, g_dtype, n * C + c) * m);
}

// ---------------------------------------------------------------------------- latent mix backward
__global__ void __launch_bounds__(256) latent_mix_bwd_kernel(const void* gz, int gz_dtype, int Cz, const float* __restrict__ q, int Cq,
                                                             const float* __restrict__ pp, const float* __restrict__ eps,
                                                             SeedArg seed_arg, int level, int64_t sample0,
                                                             const float* __restrict__ alpha_dev, float temp, int Z, int N, int H,
                                                             int W, float* __restrict__ g_q, int Cgq, float* __restrict__ g_p) {
  const uint64_t seed = seed_arg.get();
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * H * W * Cgq) return;
  const int zc = (int)(idx % Cgq);
  const int64_t pix = idx / Cgq;
  if (zc >= Z) { g_q[idx] = 0.f; return; }          // zero padding channels (tensor-core K padding)
  const int x = (int)(pix % W);
  const int y = (int)((pix / W) % H);
  const int64_t n = pix / ((int64_t)W * H);
  const float a = *alpha_dev;
  const float g = ld1b(gz, gz_dtype, pix * Cz + zc);
  const float mu_q = q[pix * Cq + zc];
  if (pp == nullptr) {
    g_q[idx] = g * (1.f - a) * sc5_grad(mu_q);
    return;
  }
  const int64_t e_idx = (((int64_t)zc) * H + y) * W + x;
  float e;
  if (eps != nullptr) e = eps[n * Z * H * W + e_idx];
  else {                                             // same stream layout as the forward kernel (latent_eps4)
    float z4[4];
    latent_eps4(seed, (uint64_t)(sample0 + n) * 64ull + (uint64_t)(level + 1), zc >> 2, y * W + x, H * W, z4);
    e = z4[zc & 3];
  }
  const float mu_p = pp[pix * 2 * Z + zc], ls_p = pp[pix * 2 * Z + Z + zc];
  const float d_enc = (1.f - a) * sc5_grad(mu_p + mu_q);
  g_q[idx] = g * d_enc;
  g_p[pix * 2 * Z + zc] = g * (d_enc + a * sc5_grad(mu_p));
  g_p[pix * 2 * Z + Z + zc] = g * a * e * temp * expf(softclamp5_(ls_p)) * sc5_grad(ls_p);
}

// 4 channels per thread (all channel counts multiples of 4): one Philox call per 4 channels instead of four, 16-byte accesses
__global__ void __launch_bounds__(256) latent_mix_bwd_vec4_kernel(const void* gz, int gz_dtype, int Cz, const float* __restrict__ q, int Cq,
                                                                  const float* __restrict__ pp, const float* __restrict__ eps,
                                                                  SeedArg seed_arg, int level, int64_t sample0,
                                                                  const float* __restrict__ alpha_dev, float temp, int Z, int N, int H,
                                                                  int W, float* __restrict__ g_q, int Cgq, float* __restrict__ g_p) {
  const uint64_t seed = seed_arg.get();
  const int groups = Cgq >> 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * H * W * groups) return;
  const int zc = (int)(idx % groups) * 4;
  const int64_t pix = idx / groups;
  float4* gq4 = reinterpret_cast<float4*>(g_q + pix * Cgq + zc);
  if (zc >= Z) { *gq4 = make_float4(0.f, 0.f, 0.f, 0.f); return; }       // zero padding channels (tensor-core K padding)
  const int x = (int)(pix % W);
  const int y = (int)((pix / W) % H);
  const int64_t n = pix / ((int64_t)W * H);
  const float a = *alpha_dev;
  float g[4], mq[4];
  if (gz_dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(gz) + pix * Cz + zc, g);
  else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(gz) + pix * Cz + zc, g);
  ld4<float>(q + pix * Cq + zc, mq);
  if (pp == nullptr) {
    *gq4 = make_float4(g[0] * (1.f - a) * sc5_grad(mq[0]), g[1] * (1.f - a) * sc5_grad(mq[1]), g[2] * (1.f - a) * sc5_grad(mq[2]),
                       g[3] * (1.f - a) * sc5_grad(mq[3]));
    return;
  }
  float e[4];
  if (eps != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) e[j] = eps[n * Z * H * W + (((int64_t)(zc + j)) * H + y) * W + x];
  } else {
    latent_eps4(seed, (uint64_t)(sample0 + n) * 64ull + (uint64_t)(level + 1), zc >> 2, y * W + x, H * W, e);
  }
  float mp[4], lp[4], o_q[4], o_m[4], o_l[4];
  ld4<float>(pp + pix * 2 * Z + zc, mp);
  ld4<float>(pp + pix * 2 * Z + Z + zc, lp);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float d_enc = (1.f - a) * sc5_grad(mp[j] + mq[j]);
    o_q[j] = g[j] * d_enc;
    o_m[j] = g[j] * (d_enc + a * sc5_grad(mp[j]));
    o_l[j] = g[j] * a * e[j] * temp * expf(softclamp5_(lp[j])) * sc5_grad(lp[j]);
  }
  *gq4 = make_float4(o_q[0], o_q[1], o_q[2], o_q[3]);
  st4<float>(g_p + pix * 2 * Z + zc, o_m);
  st4<float>(g_p + pix * 2 * Z + Z + zc, o_l);
}

// ---------------------------------------------------------------------------- DiscMixLogistic mean backward
__global__ void __launch_bounds__(128) discmix_mean_bwd_kernel(const float* __restrict__ logits, int n_mix, int HW, int64_t total_pix,
                                                               const float* __restrict__ g_pur, const void* g_cls, int gc_dtype,
                                                               float* __restrict__ g_logits, int Cg) {
  const int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= total_pix) return;
  const int CL = 10 * n_mix;
  const float* l = logits + pix * CL;
  float* gl = g_logits + pix * Cg;
  for (int c = CL; c < Cg; ++c) gl[c] = 0.f;              // channel padding (tensor-core K alignment of the dgrad conv)
  const int64_t n = pix / HW, hw = pix % HW;
  // incoming gradient w.r.t. v = (r, g, b) in [-1, 1]
  float gv[3] = {0.f, 0.f, 0.f};
  if (g_pur != nullptr) {
#pragma unroll
    for (int c = 0; c < 3; ++c) gv[c] += 0.5f * g_pur[(n * 3 + c) * HW + hw];
  }
  if (g_cls != nullptr) {
#pragma unroll
    for (int c = 0; c < 3; ++c) gv[c] += ld1b(g_cls, gc_dtype, pix * 3 + c);
  }
  float mx = l[0];
  for (int m = 1; m < n_mix; ++m) mx = fmaxf(mx, l[m]);
  float den = 0.f, mu[3] = {0.f, 0.f, 0.f}, kk[3] = {0.f, 0.f, 0.f};
  for (int m = 0; m < n_mix; ++m) {
    const float e = expf(l[m] - mx);
    const float* qd = l + n_mix + 9 * m;
    den += e;
#pragma unroll
    for (int c = 0; c < 3; ++c) { mu[c] = fmaf(e, qd[c], mu[c]); kk[c] = fmaf(e, tanhf(qd[6 + c]), kk[c]); }
  }
  const float inv = 1.f / den;
#pragma unroll
  for (int c = 0; c < 3; ++c) { mu[c] *= inv; kk[c] *= inv; }
  const float r_pre = mu[0];
  const float r = fminf(fmaxf(r_pre, -1.f), 1.f);
  const float g_pre = fmaf(kk[0], r, mu[1]);
  const float g = fminf(fmaxf(g_pre, -1.f), 1.f);
  const float b_pre = mu[2] + kk[1] * r + kk[2] * g;
  // clamp backward (inclusive bounds, torch semantics)
  const float gb = (b_pre >= -1.f && b_pre <= 1.f) ? gv[2] : 0.f;
  float g_mu[3], g_k[3];
  g_mu[2] = gb; g_k[1] = gb * r; g_k[2] = gb * g;
  float gr_acc = gv[0] + gb * kk[1];
  float gg_acc = gv[1] + gb * kk[2];
  const float gg = (g_pre >= -1.f && g_pre <= 1.f) ? gg_acc : 0.f;
  g_mu[1] = gg; g_k[0] = gg * r;
  gr_acc += gg * kk[0];
  g_mu[0] = (r_pre >= -1.f && r_pre <= 1.f) ? gr_acc : 0.f;
  // through the mixture weights
  float dot = 0.f;
  for (int m = 0; m < n_mix; ++m) {
    const float pi = expf(l[m] - mx) * inv;
    const float* qd = l + n_mix + 9 * m;
    float gpi = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float th = tanhf(qd[6 + c]);
      gpi += qd[c] * g_mu[c] + th * g_k[c];
      gl[n_mix + 9 * m + c] = pi * g_mu[c];
      gl[n_mix + 9 * m + 3 + c] = 0.f;                      // log-scales do not reach the mean
      gl[n_mix + 9 * m + 6 + c] = pi * (1.f - th * th) * g_k[c];
    }
    gl[m] = gpi;                                            // temporarily d/d pi_m
    dot = fmaf(pi, gpi, dot);
  }
  for (int m = 0; m < n_mix; ++m) {
    const float pi = expf(l[m] - mx) * inv;
    gl[m] = pi * (gl[m] - dot);
  }
}

// same arithmetic, but the 100 logits of a pixel (400-byte rows) go through shared memory: the per-pixel kernel above issues 100 scalar
// loads / 104 scalar stores whose 32 lanes hit 32 different lines (L1-wavefront bound: 1.9 ms at batch 512, 7x the HBM time)
__global__ void __launch_bounds__(128) discmix_mean_bwd_smem_kernel(const float* __restrict__ logits, int n_mix, int HW, int64_t total_pix,
                                                                    const float* __restrict__ g_pur, const void* g_cls, int gc_dtype,
                                                                    float* __restrict__ g_logits, int Cg, int stride) {
  extern __shared__ float s_row[];                       // [128][stride], stride odd >= Cg: conflict-free rows, updated in place
  const int CL = 10 * n_mix;
  const int64_t pix0 = (int64_t)blockIdx.x * 128;
  const int npix = (int)min((int64_t)128, total_pix - pix0);
  for (int i = threadIdx.x; i < npix * CL; i += 128) {
    const int p = i / CL;
    s_row[p * stride + (i - p * CL)] = __ldg(logits + pix0 * CL + i);
  }
  __syncthreads();
  if ((int)threadIdx.x < npix) {
    const int64_t pix = pix0 + threadIdx.x;
    float* l = s_row + threadIdx.x * stride;             // reads logits, ends up holding d loss / d logits
    for (int c = CL; c < Cg; ++c) l[c] = 0.f;
    const int64_t n = pix / HW, hw = pix % HW;
    float gv[3] = {0.f, 0.f, 0.f};
    if (g_pur != nullptr) {
#pragma unroll
      for (int c = 0; c < 3; ++c) gv[c] += 0.5f * g_pur[(n * 3 + c) * HW + hw];
    }
    if (g_cls != nullptr) {
#pragma unroll
      for (int c = 0; c < 3; ++c) gv[c] += ld1b(g_cls, gc_dtype, pix * 3 + c);
    }
    float mx = l[0];
    for (int m = 1; m < n_mix; ++m) mx = fmaxf(mx, l[m]);
    float den = 0.f, mu[3] = {0.f, 0.f, 0.f}, kk[3] = {0.f, 0.f, 0.f};
    for (int m = 0; m < n_mix; ++m) {
      const float e = expf(l[m] - mx);
      const float* qd = l + n_mix + 9 * m;
      den += e;
#pragma unroll
      for (int c = 0; c < 3; ++c) { mu[c] = fmaf(e, qd[c], mu[c]); kk[c] = fmaf(e, tanhf(qd[6 + c]), kk[c]); }
    }
    const float inv = 1.f / den;
#pragma unroll
    for (int c = 0; c < 3; ++c) { mu[c] *= inv; kk[c] *= inv; }
    const float r_pre = mu[0];
    const float r = fminf(fmaxf(r_pre, -1.f), 1.f);
    const float g_pre = fmaf(kk[0], r, mu[1]);
    const float g = fminf(fmaxf(g_pre, -1.f), 1.f);
    const float b_pre = mu[2] + kk[1] * r + kk[2] * g;
    const float gb = (b_pre >= -1.f && b_pre <= 1.f) ? gv[2] : 0.f;
    float g_mu[3], g_k[3];
    g_mu[2] = gb; g_k[1] = gb * r; g_k[2] = gb * g;
    float gr_acc = gv[0] + gb * kk[1];
    const float gg_acc = gv[1] + gb * kk[2];
    const float gg = (g_pre >= -1.f && g_pre <= 1.f) ? gg_acc : 0.f;
    g_mu[1] = gg; g_k[0] = gg * r;
    gr_acc += gg * kk[0];
    g_mu[0] = (r_pre >= -1.f && r_pre <= 1.f) ? gr_acc : 0.f;
    float dot = 0.f;
    for (int m = 0; m < n_mix; ++m) {
      const float pi = expf(l[m] - mx) * inv;
      float* qd = l + n_mix + 9 * m;
      float gpi = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float q = qd[c], th = tanhf(qd[6 + c]);
        gpi += q * g_mu[c] + th * g_k[c];
        qd[c] = pi * g_mu[c];
        qd[6 + c] = pi * (1.f - th * th) * g_k[c];
      }
      qd[3] = pi;                                          // stash (the log-scale slots end up zero)
      qd[4] = 0.f; qd[5] = 0.f;
      l[m] = gpi;                                          // temporarily d / d pi_m
      dot = fmaf(pi, gpi, dot);
    }
    for (int m = 0; m < n_mix; ++m) {
      float* qd = l + n_mix + 9 * m;
      l[m] = qd[3] * (l[m] - dot);
      qd[3] = 0.f;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < npix * Cg; i += 128) {
    const int p = i / Cg;
    g_logits[pix0 * Cg + i] = s_row[p * stride + (i - p * Cg)];
  }
}

static int pix_per_block_se(int HW) { return HW < 128 ? HW : 128; }

}  // namespace ga

using namespace ga;

extern "C" int ga_affine_act_bwd(const ga_tensor* g, const ga_tensor* x, const float* scale, const float* shift, int act,
                                 const ga_tensor* add, const ga_tensor* out, void* stream) {
  GA_CHECK(g && x && out && same_shape(g, x) && same_shape(g, out), "ga_affine_act_bwd: shape mismatch");
  GA_CHECK((scale == nullptr) == (shift == nullptr), "ga_affine_act_bwd: scale and shift go together");
  GA_CHECK(!add || same_shape(add, out), "ga_affine_act_bwd: add shape mismatch");
  const int64_t total = numel(g);
  if (total == 0) return 0;
  if ((g->c & 3) == 0)
    affine_act_bwd_vec4_kernel<<<cdiv(total / 4, 256), 256, 0, (cudaStream_t)stream>>>(g->data, g->dtype, x->data, x->dtype, scale, shift, act,
                                                                                       add ? add->data : nullptr, add ? add->dtype : GA_F32,
                                                                                       out->data, out->dtype, g->c, total / 4);
  else
    affine_act_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(g->data, g->dtype, x->data, x->dtype, scale, shift, act,
                                                                              add ? add->data : nullptr, add ? add->dtype : GA_F32,
                                                                              out->data, out->dtype, g->c, total);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_add(const ga_tensor* a, const ga_tensor* b, const ga_tensor* out, void* stream) {
  GA_CHECK(a && b && out && same_shape(a, b) && same_shape(a, out), "ga_add: shape mismatch");
  const int64_t total = numel(a);
  if (total == 0) return 0;
  if (a->dtype == GA_F32 && b->dtype == GA_F32 && out->dtype == GA_F32 && (total & 3) == 0 &&
      ((((uintptr_t)a->data) | ((uintptr_t)b->data) | ((uintptr_t)out->data)) & 15) == 0) {
    add_f32x4_kernel<<<(unsigned)cdiv(total / 4, 1024), 256, 0, (cudaStream_t)stream>>>((const float4*)a->data, (const float4*)b->data,
                                                                                         (float4*)out->data, total / 4);
    GA_LAUNCH_OK();
    return 0;
  }
  add_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(a->data, a->dtype, b->data, b->dtype, out->data, out->dtype, total);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_se_residual_bwd(const ga_tensor* g_out, const ga_tensor* r, const float* sums, float* dots_ws, const float* w1,
                                  const float* b1, const float* w2, const float* b2, int hidden, float res_scale,
                                  const ga_tensor* g_r, void* stream) {
  GA_CHECK(g_out && r && sums && dots_ws && w1 && w2 && g_r, "ga_se_residual_bwd: null argument");
  GA_CHECK(same_shape(g_out, r) && same_shape(g_out, g_r), "ga_se_residual_bwd: shape mismatch");
  if (numel(r) == 0) return 0;
  const int HW = r->h * r->w, C = r->c;
  const int ppb = pix_per_block_se(HW);
  const int nparts = cdiv(HW, ppb);
  cudaStream_t s = (cudaStream_t)stream;
  se_bwd_reduce_kernel<<<dim3(nparts, r->n), 256, 0, s>>>(g_out->data, g_out->dtype, r->data, r->dtype, HW, C, ppb, dots_ws);
  GA_LAUNCH_OK();
  SeBwdParams p;
  p.g = g_out->data; p.g_dtype = g_out->dtype; p.sums = sums; p.dots = dots_ws;
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.hidden = hidden; p.res_scale = res_scale;
  // the apply stage recomputes the gate MLP and its backward per CTA (five block-wide phases): give a CTA up to 512 pixels of an image so that
  // the preamble is paid 4x less often at 32x32 (the slicing of the SUMS stays 128 pixels: nparts)
  static int apply_ppb_max = -1;
  if (apply_ppb_max < 0) { const char* e = getenv("GA_SE_BWD_APPLY_PPB"); apply_ppb_max = e ? atoi(e) : 512; }
  const int appb = HW < apply_ppb_max ? HW : apply_ppb_max;
  p.g_r = g_r->data; p.gr_dtype = g_r->dtype; p.HW = HW; p.C = C; p.pix_per_block = appb; p.nparts = nparts;
  const size_t smem = (4 * (size_t)C + 2 * hidden) * sizeof(float);
  GA_CHECK(smem <= 48 * 1024, "ga_se_residual_bwd: too many channels");
  se_bwd_apply_kernel<<<dim3(cdiv(HW, appb), r->n), 256, smem, s>>>(p);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_sumpool2x2(const ga_tensor* in, const ga_tensor* mul, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && in->h == 2 * out->h && in->w == 2 * out->w && in->c == out->c && in->n == out->n, "ga_sumpool2x2: shape mismatch");
  GA_CHECK(!mul || same_shape(mul, out), "ga_sumpool2x2: mul shape mismatch");
  const int64_t total = numel(out);
  if (total == 0) return 0;
  if ((out->c & 3) == 0 && ((((uintptr_t)in->data) | ((uintptr_t)out->data) | (mul ? (uintptr_t)mul->data : 0)) & 15) == 0) {
    sumpool2x2_vec4_kernel<<<cdiv(total / 4, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, mul ? mul->data : nullptr,
                                                                                  mul ? mul->dtype : GA_F32, out->data, out->dtype, total / 4,
                                                                                  out->h, out->w, out->c);
    GA_LAUNCH_OK();
    return 0;
  }
  sumpool2x2_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, mul ? mul->data : nullptr,
                                                                        mul ? mul->dtype : GA_F32, out->data, out->dtype, out->n, out->h,
                                                                        out->w, out->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_depth_to_space2(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && in->dtype == GA_F32 && out->dtype == GA_F32, "ga_depth_to_space2: fp32 tensors expected");
  GA_CHECK(out->n == in->n && out->h == 2 * in->h && out->w == 2 * in->w && in->c == 4 * out->c && out->c % 4 == 0,
           "ga_depth_to_space2: shape mismatch (in [n,h,w,4c] -> out [n,2h,2w,c], c % 4 == 0)");
  const int64_t total4 = numel(out) / 4;
  if (total4 == 0) return 0;
  depth_to_space2_kernel<<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>((const float4*)in->data, (float4*)out->data, total4, in->h,
                                                                              in->w, out->c / 4);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_phase_interleave(const ga_tensor* in, const ga_tensor* add, const ga_tensor* mul, int mul_mode, const float* slope,
                                   const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && in->dtype == GA_F32, "ga_phase_interleave: fp32 input expected");
  GA_CHECK(out->n == in->n && out->h == 2 * in->h && out->w == 2 * in->w && in->c == 4 * out->c && out->c % 4 == 0,
           "ga_phase_interleave: shape mismatch (in [n,h,w,4c] -> out [n,2h,2w,c], c % 4 == 0)");
  GA_CHECK(!add || same_shape(add, out), "ga_phase_interleave: add shape mismatch");
  GA_CHECK(!mul || same_shape(mul, out), "ga_phase_interleave: mul shape mismatch");
  GA_CHECK(!mul || mul_mode != GA_MUL_PRELU_FROM_Y || slope, "ga_phase_interleave: PReLU mask needs slope");
  auto aligned = [](const ga_tensor* t) { return !t || (((uintptr_t)t->data) & (t->dtype == GA_F32 ? 15 : 7)) == 0; };
  GA_CHECK(aligned(in) && aligned(out) && aligned(add) && aligned(mul), "ga_phase_interleave: tensors must be 4-channel-vector aligned");
  const int64_t total4 = numel(out) / 4;
  if (total4 == 0) return 0;
  const int ad = add ? add->dtype : GA_F32, md = mul ? mul->dtype : GA_F32;
  if (out->dtype == GA_F32)
    phase_interleave_kernel<float><<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(
        (const float4*)in->data, add ? add->data : nullptr, ad, mul ? mul->data : nullptr, md, mul_mode, slope, (float*)out->data, total4, in->h,
        in->w, out->c / 4);
  else
    phase_interleave_kernel<__nv_bfloat16><<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(
        (const float4*)in->data, add ? add->data : nullptr, ad, mul ? mul->data : nullptr, md, mul_mode, slope, (__nv_bfloat16*)out->data, total4,
        in->h, in->w, out->c / 4);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_subsample2x_bwd(const ga_tensor* g, const ga_tensor* out, void* stream) {
  GA_CHECK(g && out && g->n == out->n && g->c == out->c && g->h == (out->h + 1) / 2 && g->w == (out->w + 1) / 2 && out->c % 4 == 0,
           "ga_subsample2x_bwd: shape mismatch (g [n,ceil(h/2),ceil(w/2),c] -> out [n,h,w,c], c % 4 == 0)");
  const int64_t total4 = numel(out) / 4;
  if (total4 == 0) return 0;
  subsample2x_bwd_kernel<<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(g->data, g->dtype, out->data, out->dtype, total4, out->h, out->w,
                                                                              out->c / 4, g->h, g->w);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_upsample_bilinear2x_bwd(const ga_tensor* g_out, const ga_tensor* g_in, void* stream) {
  GA_CHECK(g_out && g_in && g_out->h == 2 * g_in->h && g_out->w == 2 * g_in->w && g_out->c == g_in->c && g_out->n == g_in->n,
           "ga_upsample_bilinear2x_bwd: shape mismatch");
  const int64_t total = numel(g_in);
  if (total == 0) return 0;
  bilinear2x_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(g_out->data, g_out->dtype, g_in->data, g_in->dtype, g_in->n,
                                                                            g_in->h, g_in->w, g_in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_maxpool2x2_bwd(const ga_tensor* x_in, const ga_tensor* g_out, int relu, const ga_tensor* g_in, void* stream) {
  GA_CHECK(x_in && g_out && g_in && same_shape(x_in, g_in) && g_out->h == x_in->h / 2 && g_out->w == x_in->w / 2 &&
               g_out->c == x_in->c && g_out->n == x_in->n && (x_in->h % 2 == 0) && (x_in->w % 2 == 0),
           "ga_maxpool2x2_bwd: shape mismatch");
  const int64_t total = numel(g_out);
  if (total == 0) return 0;
  maxpool2x2_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x_in->data, x_in->dtype, g_out->data, g_out->dtype, relu,
                                                                            g_in->data, g_in->dtype, x_in->n, x_in->h, x_in->w, x_in->c);
  GA_LAUNCH_OK();
  return 0;
}


extern "C" int ga_maxpool3x3s2_bwd(const ga_tensor* x_in, const ga_tensor* g_out, int relu, const ga_tensor* g_in, void* stream) {
  GA_CHECK(x_in && g_out && g_in && same_shape(x_in, g_in) && g_out->h == (x_in->h - 1) / 2 + 1 && g_out->w == (x_in->w - 1) / 2 + 1 &&
               g_out->c == x_in->c && g_out->n == x_in->n, "ga_maxpool3x3s2_bwd: shape mismatch");
  const int64_t total = numel(x_in);
  if (total == 0) return 0;
  maxpool3x3s2_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x_in->data, x_in->dtype, g_out->data, g_out->dtype, relu,
                                                                              g_in->data, g_in->dtype, x_in->n, x_in->h, x_in->w, x_in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_avgpool_bwd_relu(const ga_tensor* g_feat, const ga_tensor* y, const ga_tensor* g_in, void* stream) {
  GA_CHECK(g_feat && y && g_in && same_shape(y, g_in) && g_feat->n == y->n && g_feat->c == y->c && g_feat->h == 1 && g_feat->w == 1,
           "ga_avgpool_bwd_relu: shape mismatch");
  const int64_t total = numel(y);
  if (total == 0) return 0;
  avgpool_bwd_relu_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(g_feat->data, g_feat->dtype, y->data, y->dtype, g_in->data,
                                                                              g_in->dtype, y->h * y->w, y->c, total);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_latent_mix_bwd(const ga_tensor* g_z, const ga_tensor* q, const ga_tensor* p, const float* eps, uint64_t seed,
                                 int level, int64_t sample0, const float* alpha_dev, float temperature, int zdim,
                                 const ga_tensor* g_q, const ga_tensor* g_p, void* stream) {
  GA_CHECK(g_z && q && g_q && alpha_dev, "ga_latent_mix_bwd: null argument");
  GA_CHECK(q->dtype == GA_F32 && g_q->dtype == GA_F32 && g_q->c >= zdim, "ga_latent_mix_bwd: q / g_q must be fp32, g_q with >= zdim channels");
  GA_CHECK((p == nullptr) == (g_p == nullptr), "ga_latent_mix_bwd: p and g_p go together");
  GA_CHECK(!p || (p->dtype == GA_F32 && g_p->dtype == GA_F32 && p->c == 2 * zdim && g_p->c == 2 * zdim), "ga_latent_mix_bwd: p / g_p must be fp32 with 2*zdim channels");
  const int64_t total = (int64_t)q->n * q->h * q->w * g_q->c;
  if (total == 0) return 0;
  if ((zdim & 3) == 0 && (g_z->c & 3) == 0 && (q->c & 3) == 0 && (g_q->c & 3) == 0 &&
      ((((uintptr_t)g_z->data) | ((uintptr_t)q->data) | ((uintptr_t)g_q->data) | (p ? (uintptr_t)p->data : 0) | (g_p ? (uintptr_t)g_p->data : 0)) & 15) == 0) {
    const int64_t total4 = (int64_t)q->n * q->h * q->w * (g_q->c / 4);
    latent_mix_bwd_vec4_kernel<<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(
        g_z->data, g_z->dtype, g_z->c, (const float*)q->data, q->c, p ? (const float*)p->data : nullptr, eps, make_seed(seed, (cudaStream_t)stream), level, sample0,
        alpha_dev, temperature, zdim, q->n, q->h, q->w, (float*)g_q->data, g_q->c, g_p ? (float*)g_p->data : nullptr);
    GA_LAUNCH_OK();
    return 0;
  }
  latent_mix_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(
      g_z->data, g_z->dtype, g_z->c, (const float*)q->data, q->c, p ? (const float*)p->data : nullptr, eps, make_seed(seed, (cudaStream_t)stream), level, sample0,
      alpha_dev, temperature, zdim, q->n, q->h, q->w, (float*)g_q->data, g_q->c, g_p ? (float*)g_p->data : nullptr);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_discmix_mean_bwd(const ga_tensor* logits, int n_mix, const float* g_purified_nchw, const ga_tensor* g_cls,
                                   const ga_tensor* g_logits, void* stream) {
  GA_CHECK(logits && g_logits && logits->n == g_logits->n && logits->h == g_logits->h && logits->w == g_logits->w &&
               g_logits->c >= logits->c && logits->dtype == GA_F32 && g_logits->dtype == GA_F32,
           "ga_discmix_mean_bwd: logits / g_logits must be fp32 tensors of the same spatial shape (g_logits may be channel-padded)");
  GA_CHECK(logits->c == 10 * n_mix, "ga_discmix_mean_bwd: logits must have 10*n_mix channels");
  GA_CHECK(g_purified_nchw || g_cls, "ga_discmix_mean_bwd: no incoming gradient");
  const int64_t total_pix = (int64_t)logits->n * logits->h * logits->w;
  if (total_pix == 0) return 0;
  {
    const int stride = g_logits->c | 1;
    const int smem = 128 * stride * (int)sizeof(float);
    static int configured = 0;
    if (smem <= 200 * 1024) {
      if (configured < smem) {
        GA_CUDA(cudaFuncSetAttribute(discmix_mean_bwd_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = smem;
      }
      discmix_mean_bwd_smem_kernel<<<cdiv(total_pix, 128), 128, smem, (cudaStream_t)stream>>>(
          (const float*)logits->data, n_mix, logits->h * logits->w, total_pix, g_purified_nchw, g_cls ? g_cls->data : nullptr,
          g_cls ? g_cls->dtype : GA_F32, (float*)g_logits->data, g_logits->c, stride);
      GA_LAUNCH_OK();
      return 0;
    }
  }
  discmix_mean_bwd_kernel<<<cdiv(total_pix, 128), 128, 0, (cudaStream_t)stream>>>(
      (const float*)logits->data, n_mix, logits->h * logits->w, total_pix, g_purified_nchw, g_cls ? g_cls->data : nullptr,
      g_cls ? g_cls->dtype : GA_F32, (float*)g_logits->data, g_logits->c);
  GA_LAUNCH_OK();
  return 0;
}
