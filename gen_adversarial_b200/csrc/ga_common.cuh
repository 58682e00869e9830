// Shared device/host helpers for libga_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/ga_b200.h"

namespace ga {

// ----------------------------------------------------------------------------- host-side error plumbing
void set_error(const char* fmt, ...);
void count_launch();

#define GA_CHECK(cond, ...)                         \
  do {                                              \
    if (!(cond)) {                                  \
      ::ga::set_error(__VA_ARGS__);                 \
      return 1;                                     \
    }                                               \
  } while (0)

#define GA_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ::ga::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, cudaGetErrorName(_e), \
                      cudaGetErrorString(_e));                                          \
      return 2;                                                                         \
    }                                                                                   \
  } while (0)

// call after every kernel launch
#define GA_LAUNCH_OK()                 \
  do {                                 \
    ::ga::count_launch();              \
    GA_CUDA(cudaPeekAtLastError());    \
  } while (0)

static inline int64_t numel(const ga_tensor* t) { return (int64_t)t->n * t->h * t->w * t->c; }
static inline bool same_shape(const ga_tensor* a, const ga_tensor* b) {
  return a->n == b->n && a->h == b->h && a->w == b->w && a->c == b->c;
}
static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ----------------------------------------------------------------------------- device math
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float siluf_(float x) { return x / (1.0f + expf(-x)); }
__device__ __forceinline__ float eluf_(float x) { return x > 0.0f ? x : expm1f(x); }
__device__ __forceinline__ float softclamp5_(float x) { return 5.0f * tanhf(x * 0.2f); }
// one latent channel of a level with a prior (models.py:198-206,243-250):
//   z = (1-a) * sc(mu_p + mu_q) + a * (sc(mu_p) + eps * T * exp(sc(logsig_p)))
// shared by latent_mix (elementwise.cu) and the fused level tail (latent_level.cu) so both round identically
__device__ __forceinline__ float latent_mix_prior(float a, float mq, float mp, float lp, float e, float temp) {
  return (1.f - a) * softclamp5_(mp + mq) + a * (softclamp5_(mp) + e * (temp * expf(softclamp5_(lp))));
}

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case GA_ACT_SILU: return siluf_(v);
    case GA_ACT_ELU: return eluf_(v);
    case GA_ACT_RELU: return fmaxf(v, 0.0f);
    case GA_ACT_LRELU_SQRT2: return (v > 0.0f ? v : 0.2f * v) * 1.4142135623730951f;
    default: return v;
  }
}
// activation with per-channel slope (PReLU); other codes ignore `slope`
__device__ __forceinline__ float apply_act_s(float v, int act, float slope) {
  return act == GA_ACT_PRELU ? (v > 0.0f ? v : slope * v) : apply_act(v, act);
}
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// SiLU with ONE transcendental (MUFU.TANH): v * sigmoid(v) = v * (0.5 * tanh(v/2) + 0.5); abs error ~5e-4 * |v|, far
// below bf16 rounding (4e-3 * |v|) -- used only where the result is rounded to bf16
__device__ __forceinline__ float silu_fast(float v) {
  const float h = 0.5f * v;
  return fmaf(h, tanh_approx(h), h);
}
// fast-math variant for bf16 outputs
__device__ __forceinline__ float apply_act_fast(float v, int act) {
  switch (act) {
    case GA_ACT_SILU: return silu_fast(v);
    case GA_ACT_ELU: return v > 0.0f ? v : __expf(v) - 1.0f;
    case GA_ACT_RELU: return fmaxf(v, 0.0f);
    case GA_ACT_LRELU_SQRT2: return (v > 0.0f ? v : 0.2f * v) * 1.4142135623730951f;
    default: return v;
  }
}
// derivative of act w.r.t. its pre-activation input v
__device__ __forceinline__ float act_grad(float v, int act) {
  switch (act) {
    case GA_ACT_SILU: {
      float s = sigmoidf_(v);
      return s * (1.0f + v * (1.0f - s));
    }
    case GA_ACT_ELU: return v > 0.0f ? 1.0f : expf(v);
    case GA_ACT_RELU: return v > 0.0f ? 1.0f : 0.0f;
    case GA_ACT_LRELU_SQRT2: return (v > 0.0f ? 1.0f : 0.2f) * 1.4142135623730951f;
    default: return 1.0f;
  }
}

// Array forms with the activation switch OUTSIDE the element loop.  A per-element `switch (act)` over five activations compiles
// to an indexed jump (BRX) per element -- measured +25..60% on the tensor-core conv epilogue -- so every vector path goes
// through these: one uniform branch per register tile, straight-line code per element.
template <int N>
__device__ __forceinline__ void apply_act_n(float (&v)[N], int act) {
  switch (act) {
    case GA_ACT_SILU:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = siluf_(v[j]);
      break;
    case GA_ACT_ELU:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = eluf_(v[j]);
      break;
    case GA_ACT_RELU:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = fmaxf(v[j], 0.0f);
      break;
    case GA_ACT_LRELU_SQRT2:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = (v[j] > 0.0f ? v[j] : 0.2f * v[j]) * 1.4142135623730951f;
      break;
    default: break;
  }
}
template <int N>
__device__ __forceinline__ void apply_act_fast_n(float (&v)[N], int act) {
  switch (act) {
    case GA_ACT_SILU:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = silu_fast(v[j]);
      break;
    case GA_ACT_ELU:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = v[j] > 0.0f ? v[j] : __expf(v[j]) - 1.0f;
      break;
    case GA_ACT_RELU:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = fmaxf(v[j], 0.0f);
      break;
    case GA_ACT_LRELU_SQRT2:
#pragma unroll
      for (int j = 0; j < N; ++j) v[j] = (v[j] > 0.0f ? v[j] : 0.2f * v[j]) * 1.4142135623730951f;
      break;
    default: break;
  }
}
// d[j] = act'(pre[j])
template <int N>
__device__ __forceinline__ void act_grad_n(const float (&pre)[N], float (&d)[N], int act) {
  switch (act) {
    case GA_ACT_SILU:
#pragma unroll
      for (int j = 0; j < N; ++j) { const float s = sigmoidf_(pre[j]); d[j] = s * (1.0f + pre[j] * (1.0f - s)); }
      break;
    case GA_ACT_ELU:
#pragma unroll
      for (int j = 0; j < N; ++j) d[j] = pre[j] > 0.0f ? 1.0f : expf(pre[j]);
      break;
    case GA_ACT_RELU:
#pragma unroll
      for (int j = 0; j < N; ++j) d[j] = pre[j] > 0.0f ? 1.0f : 0.0f;
      break;
    case GA_ACT_LRELU_SQRT2:
#pragma unroll
      for (int j = 0; j < N; ++j) d[j] = (pre[j] > 0.0f ? 1.0f : 0.2f) * 1.4142135623730951f;
      break;
    default:
#pragma unroll
      for (int j = 0; j < N; ++j) d[j] = 1.0f;
      break;
  }
}

// bf16-grade derivative (results rounded to bf16 by the caller): SiLU' from ONE MUFU.TANH -- with h = v/2, t = tanh(h):
// silu'(v) = s (1 + v (1 - s)), s = (1 + t)/2  =  1/2 + (t + h (1 - t^2)) / 2.  The exact form costs an expf and a full-precision
// division per element (~25 instructions), which made the taping epilogues of the attack path issue-bound.
template <int N>
__device__ __forceinline__ void act_grad_fast_n(const float (&pre)[N], float (&d)[N], int act) {
  if (act == GA_ACT_SILU) {
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const float h = 0.5f * pre[j];
      const float t = tanh_approx(h);
      d[j] = fmaf(0.5f, fmaf(h, fmaf(-t, t, 1.0f), t), 0.5f);
    }
  } else if (act == GA_ACT_ELU) {
#pragma unroll
    for (int j = 0; j < N; ++j) d[j] = pre[j] > 0.0f ? 1.0f : __expf(pre[j]);
  } else {
    act_grad_n<N>(pre, d, act);
  }
}

// SiLU and its derivative from the SAME MUFU.TANH (taping epilogues: the XU pipe does 16 lanes / clk / SM, a second tanh per element
// would cost as much as the whole HBM time of a 6C-wide 1x1 conv)
template <int N>
__device__ __forceinline__ void silu_with_grad_fast_n(const float (&pre)[N], float (&y)[N], float (&d)[N]) {   // y may alias pre
#pragma unroll
  for (int j = 0; j < N; ++j) {
    const float h = 0.5f * pre[j];
    const float t = tanh_approx(h);
    y[j] = fmaf(h, t, h);
    d[j] = fmaf(0.5f, fmaf(h, fmaf(-t, t, 1.0f), t), 0.5f);
  }
}

// packed fp32 FMA (Blackwell FFMA2): two independent FMAs per issue slot -- d.xy = a.xy * b.xy + c.xy
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(d)
      : "l"(*reinterpret_cast<uint64_t*>(&a)), "l"(*reinterpret_cast<uint64_t*>(&b)), "l"(*reinterpret_cast<uint64_t*>(&c)));
  return *reinterpret_cast<float2*>(&d);
}

// slope: PReLU slope of m's channel (GA_MUL_PRELU_FROM_Y only)
__device__ __forceinline__ float mul_factor(float m, int mode, float slope) {
  switch (mode) {
    case GA_MUL_RELU_MASK: return m > 0.0f ? 1.0f : 0.0f;
    case GA_MUL_ELU_FROM_Y: return m > 0.0f ? 1.0f : m + 1.0f;
    case GA_MUL_PRELU_FROM_Y: return m > 0.0f ? 1.0f : slope;
    default: return m;
  }
}

// ----------------------------------------------------------------------------- typed loads / stores
template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// 4 consecutive elements (16-byte fp32 / 8-byte bf16); caller guarantees alignment
template <typename T> __device__ __forceinline__ void ld4(const T* p, float (&v)[4]);
template <> __device__ __forceinline__ void ld4<float>(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <> __device__ __forceinline__ void ld4<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[4]) {
  uint2 t = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
  v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
}
template <typename T> __device__ __forceinline__ void st4(T* p, const float (&v)[4]);
template <> __device__ __forceinline__ void st4<float>(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <> __device__ __forceinline__ void st4<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  uint2 t;
  t.x = *reinterpret_cast<uint32_t*>(&a);
  t.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = t;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 a = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&a);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ----------------------------------------------------------------------------- TF32 producers
// tcgen05 kind::tf32 TRUNCATES its fp32 operands to 10 mantissa bits; truncation is biased (every operand shrinks), and the bias
// compounds over a 50-layer backbone (measured: worse than bf16 operands).  While ga_f32_round_tf32(1) is in effect, kernels that
// write fp32 activations consumed by a TF32 conv round them to nearest (cvt.rna.tf32.f32), so the MMA's truncation is exact.
int round_tf32_enabled();                              // host: launch-time value of the switch
__device__ __forceinline__ float round_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}

// ----------------------------------------------------------------------------- seed with an optional device-side salt
// Kernels take their Philox seed by value.  Under CUDA-graph replay a by-value seed is frozen into the graph, so every replay would
// draw the same noise; when a salt buffer is registered (ga_seed_salt_set) the effective seed of CAPTURED launches is seed + *salt, and ga_seed_salt_bump
// -- a one-thread kernel captured as the first node of the graph -- advances the salt on every replay with no host involvement.
const uint64_t* seed_salt_ptr();                       // host: the registered device buffer (nullptr = none)
struct SeedArg {
  uint64_t seed;
  const uint64_t* salt;
  __device__ __forceinline__ uint64_t get() const { return salt != nullptr ? seed + *salt : seed; }
};
// The salt applies ONLY to launches recorded into a CUDA graph: an eager launch keeps its by-value seed, so (a) a fixed seed reproduces the
// same noise in eager mode whether or not a graph has run in the process, and (b) a taped eager forward and its later backward passes
// regenerate the same eps even if a graph replay advanced the salt in between (the tape stores only the by-value seed).
static inline SeedArg make_seed(uint64_t seed, cudaStream_t stream) {
  const uint64_t* salt = seed_salt_ptr();
  if (salt != nullptr) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &st) != cudaSuccess || st != cudaStreamCaptureStatusActive) salt = nullptr;
  }
  return SeedArg{seed, salt};
}

// ----------------------------------------------------------------------------- counter-based RNG (Philox4x32-10)
// Stream is keyed by (seed, stream id, element counter) so results do not depend on launch geometry or on
// how a batch is sharded over GPUs (SURVEY 8e: "per-GPU seeded eps streams keyed by global sample index").
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1, uint32_t (&out)[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// four N(0,1) draws for counter block `blk` of stream (seed, stream)
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint64_t stream, uint64_t blk, float (&z)[4]) {
  uint32_t r[4];
  philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)stream, (uint32_t)(stream >> 32), (uint32_t)seed,
                (uint32_t)(seed >> 32), r);
  const float k = 2.3283064365386963e-10f;  // 2^-32
  float u0 = ((float)r[0] + 0.5f) * k, u1 = ((float)r[1] + 0.5f) * k;
  float u2 = ((float)r[2] + 0.5f) * k, u3 = ((float)r[3] + 0.5f) * k;
  float m0 = sqrtf(-2.0f * __logf(u0)), m1 = sqrtf(-2.0f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  z[0] = m0 * c0; z[1] = m0 * s0; z[2] = m1 * c1; z[3] = m1 * s1;
}
// Philox stream id of (global sample, level slot): slot 0 is the input noise, slot L + 1 the latent noise of level L
__host__ __device__ __forceinline__ uint64_t noise_stream(int64_t sample, int level) {
  return (uint64_t)sample * 64ull + (uint64_t)level;
}
// per-level latent noise eps[zc][hw] of one sample (stream = (global sample, level)): the four channels 4j .. 4j+3 of pixel hw are
// ONE Philox block (counter j * HW + hw), so a thread that owns a pixel draws 4 channels per block with no redundant rounds
__device__ __forceinline__ void latent_eps4(uint64_t seed, uint64_t stream, int j, int hw, int HW, float (&z)[4]) {
  philox_normal4(seed, stream, (uint64_t)j * (uint64_t)HW + (uint64_t)hw, z);
}
// scalar convenience: element `idx` of the stream
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t stream, uint64_t idx) {
  float z[4];
  philox_normal4(seed, stream, idx >> 2, z);
  return z[idx & 3];
}

}  // namespace ga
