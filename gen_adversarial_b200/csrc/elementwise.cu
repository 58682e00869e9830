// Bandwidth-bound fused kernels of the purification path (forward): pre-processing, depthwise 5x5,
// squeeze-excite + residual, latent mix, DiscMixLogistic mean, resampling, PGD step, cross-entropy.
// All are HBM-bound: coalesced / vectorised accesses, one pass over each tensor, fp32 math.
#include "ga_common.cuh"

namespace ga {

// runtime-dtype 4-wide access (branch is grid-uniform)
__device__ __forceinline__ void ld4d(const void* base, int dtype, int64_t off, float (&v)[4]) {
  if (dtype == GA_F32) ld4<float>(reinterpret_cast<const float*>(base) + off, v);
  else ld4<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(base) + off, v);
}
__device__ __forceinline__ void st4d(void* base, int dtype, int64_t off, const float (&v)[4]) {
  if (dtype == GA_F32) st4<float>(reinterpret_cast<float*>(base) + off, v);
  else st4<__nv_bfloat16>(reinterpret_cast<__nv_bfloat16*>(base) + off, v);
}
__device__ __forceinline__ float ld1d(const void* base, int dtype, int64_t off) {
  return dtype == GA_F32 ? reinterpret_cast<const float*>(base)[off]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[off]);
}
__device__ __forceinline__ void st1d(void* base, int dtype, int64_t off, float v) {
  if (dtype == GA_F32) reinterpret_cast<float*>(base)[off] = v;
  else reinterpret_cast<__nv_bfloat16*>(base)[off] = __float2bfloat16_rn(v);
}

// ============================================================================ noise L2 norm pre-pass
// block-level deterministic sum: warp shuffle tree, then warp 0 adds the per-warp values in fixed order
__device__ __forceinline__ float block_sum_256(float v) {
  __shared__ float s_w[8];
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) t += s_w[i];
  return t;
}

// partial[b][blockIdx.x] = sum of squares of this block's slice (no atomics: bit-reproducible)
__global__ void noise_sumsq_kernel(const float* __restrict__ noise, int chw, float* __restrict__ sumsq) {
  const int b = blockIdx.y;
  const float4* src = reinterpret_cast<const float4*>(noise + (int64_t)b * chw);
  const int n4 = chw >> 2;
  float acc = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    float4 v = __ldg(src + i);
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0)   // tail (chw not multiple of 4)
    for (int i = (n4 << 2) + threadIdx.x; i < chw; i += blockDim.x) {
      float v = noise[(int64_t)b * chw + i];
      acc += v * v;
    }
  acc = block_sum_256(acc);
  if (threadIdx.x == 0) sumsq[(int64_t)b * gridDim.x + blockIdx.x] = acc;
}

__global__ void noise_sumsq_philox_kernel(SeedArg seed_arg, int64_t sample0, int chw, float* __restrict__ sumsq) {
  const uint64_t seed = seed_arg.get();
  const int b = blockIdx.y;
  const uint64_t stream = noise_stream(sample0 + b, 0);
  const int n4 = (chw + 3) >> 2;
  float acc = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    float z[4];
    philox_normal4(seed, stream, (uint64_t)i, z);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (i * 4 + j < chw) acc += z[j] * z[j];
  }
  acc = block_sum_256(acc);
  if (threadIdx.x == 0) sumsq[(int64_t)b * gridDim.x + blockIdx.x] = acc;
}

// ============================================================================ fused pre-processing
// tile 32 rows x 32 cols, 256 threads, each thread 4 consecutive x of one row, all channels.
constexpr int PT = 32;
constexpr int MAXR = 15;
constexpr int GA_NOISE_PARTS = 16;

__device__ __forceinline__ int reflect_idx(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

template <bool BLUR>
__global__ void __launch_bounds__(256) preprocess_fwd_kernel(
    const float* __restrict__ x, const float* __restrict__ noise, const float* __restrict__ sumsq, SeedArg seed_arg,
    int nparts, int64_t sample0, float eps, const float* __restrict__ taps, int R, int normalize, int C, int H, int W,
    void* out, int out_dtype, float* __restrict__ pre) {
  const uint64_t seed = seed_arg.get();
  __shared__ float s_in[BLUR ? (PT + 2 * MAXR) : 1][BLUR ? (PT + 2 * MAXR + 1) : 1];
  __shared__ float s_h[BLUR ? (PT + 2 * MAXR) : 1][BLUR ? (PT + 1) : 1];
  __shared__ float s_taps[2 * MAXR + 1];

  const int b = blockIdx.z;
  const int tiles_x = (W + PT - 1) / PT;
  const int ty0 = (blockIdx.x / tiles_x) * PT, tx0 = (blockIdx.x % tiles_x) * PT;
  const int tid = threadIdx.x;
  const int ly = tid >> 3, lx = (tid & 7) * 4;
  const int oy = ty0 + ly, ox = tx0 + lx;
  if (BLUR) {
    if (tid < 2 * R + 1) s_taps[tid] = taps[tid];
  }
  float scale = 0.f;
  if (eps != 0.f) {
    float ss = 0.f;
    for (int i = 0; i < nparts; ++i) ss += sumsq[(int64_t)b * nparts + i];   // fixed order
    scale = eps / sqrtf(ss);
  }

  float res[4][4];   // [channel][pixel]
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if (c >= C) break;
    const float* xp = x + ((int64_t)b * C + c) * H * W;
    float v[4];
    if (BLUR) {
      const int ext = PT + 2 * R;
      __syncthreads();
      for (int i = tid; i < ext * ext; i += 256) {
        int yy = i / ext, xx = i % ext;
        int gy = reflect_idx(ty0 + yy - R, H), gx = reflect_idx(tx0 + xx - R, W);
        // tiles hanging over the image edge (H, W not multiples of 32): clamp, results are masked later
        gy = min(max(gy, 0), H - 1); gx = min(max(gx, 0), W - 1);
        s_in[yy][xx] = __ldg(xp + (int64_t)gy * W + gx);
      }
      __syncthreads();
      for (int i = tid; i < ext * PT; i += 256) {
        int yy = i / PT, xx = i % PT;
        float a = 0.f;
        for (int t = 0; t < 2 * R + 1; ++t) a = fmaf(s_taps[t], s_in[yy][xx + t], a);
        s_h[yy][xx] = a;
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float a = 0.f;
        for (int t = 0; t < 2 * R + 1; ++t) a = fmaf(s_taps[t], s_h[ly + t][lx + j], a);
        v[j] = a;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = (oy < H && ox + j < W) ? __ldg(xp + (int64_t)oy * W + ox + j) : 0.f;
    }
    if (eps != 0.f && oy < H) {
      const int64_t e0 = ((int64_t)c * H + oy) * W + ox;   // element index inside the sample
      float z[4];
      if (noise != nullptr) {
#pragma unroll
        for (int j = 0; j < 4; ++j) z[j] = (ox + j < W) ? __ldg(noise + (int64_t)b * C * H * W + e0 + j) : 0.f;
      } else {
        if ((e0 & 3) == 0) {
          philox_normal4(seed, noise_stream(sample0 + b, 0), (uint64_t)(e0 >> 2), z);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) z[j] = philox_normal(seed, noise_stream(sample0 + b, 0), (uint64_t)(e0 + j));
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = fmaf(z[j], scale, v[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float r = fminf(fmaxf(v[j], 0.f), 1.f);
      // saved UNCLAMPED: torch's clamp backward passes the gradient where 0 <= v <= 1 (inclusive)
      if (pre != nullptr && oy < H && ox + j < W) pre[(((int64_t)b * C + c) * H + oy) * W + ox + j] = v[j];
      res[c][j] = normalize ? (r - 0.5f) * 2.0f : r;
    }
  }
  if (oy < H) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (ox + j >= W) continue;
      const int64_t o = (((int64_t)b * H + oy) * W + ox + j) * C;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < C) st1d(out, out_dtype, o + c, res[c][j]);
    }
  }
}

// Blur path with a compile-time radius (7 at 64 x 64, 12 at 128 / 256: what ops.gaussian_taps produces): taps in registers, both passes
// on 16-byte shared-memory vectors (4 outputs share one sliding window), compile-time index arithmetic in the staging loop.  The generic
// kernel above spent ~1500 instructions per thread and channel on scalar LDS + runtime-bounded loops (112 us for the 50 MB of batch 512).
template <int RT>
__global__ void __launch_bounds__(256) preprocess_blur_fast_kernel(
    const float* __restrict__ x, const float* __restrict__ noise, const float* __restrict__ sumsq, SeedArg seed_arg,
    int nparts, int64_t sample0, float eps, const float* __restrict__ taps, int normalize, int C, int H, int W,
    void* out, int out_dtype, float* __restrict__ pre) {
  constexpr int EXT = PT + 2 * RT;                 // staged rows / columns
  constexpr int PIN = (EXT + 3 + 3) & ~3;          // s_in pitch: >= EXT + 2 (window over-read), multiple of 4 floats
  constexpr int PH = PT + 4;                       // s_h pitch, multiple of 4
  constexpr int NT = 2 * RT + 1;
  const uint64_t seed = seed_arg.get();
  __shared__ __align__(16) float s_in[EXT][PIN];
  __shared__ __align__(16) float s_h[EXT][PH];
  const int b = blockIdx.z;
  const int tiles_x = (W + PT - 1) / PT;
  const int ty0 = (blockIdx.x / tiles_x) * PT, tx0 = (blockIdx.x % tiles_x) * PT;
  const int tid = threadIdx.x;
  const int ly = tid >> 3, lx = (tid & 7) * 4;
  const int oy = ty0 + ly, ox = tx0 + lx;
  float tp[NT];
#pragma unroll
  for (int t = 0; t < NT; ++t) tp[t] = __ldg(taps + t);
  // reflect-border source offsets of the staged rows / columns, computed once per CTA (the staging loop is then 2 LDS + 1 LDG per element)
  __shared__ int s_gy[EXT], s_gx[EXT];
  static_assert(EXT <= 64, "index tables are filled by threads 0..EXT-1 and 64..64+EXT-1");
  if (tid < EXT) s_gy[tid] = min(max(reflect_idx(ty0 + tid - RT, H), 0), H - 1) * W;       // tiles hanging over the edge: clamped, masked later
  else if (tid >= 64 && tid < 64 + EXT) s_gx[tid - 64] = min(max(reflect_idx(tx0 + tid - 64 - RT, W), 0), W - 1);
  float scale = 0.f;
  if (eps != 0.f) {
    float ss = 0.f;
    for (int i = 0; i < nparts; ++i) ss += sumsq[(int64_t)b * nparts + i];   // fixed order
    scale = eps / sqrtf(ss);
  }
  float res[4][4];   // [channel][pixel]
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if (c >= C) break;
    const float* xp = x + ((int64_t)b * C + c) * H * W;
    __syncthreads();
    for (int i = tid; i < EXT * EXT; i += 256) {
      const int yy = i / EXT, xx = i - yy * EXT;
      s_in[yy][xx] = __ldg(xp + s_gy[yy] + s_gx[xx]);
    }
    __syncthreads();
    // horizontal pass: one item = 4 consecutive outputs of one staged row (window of 4 + 2 RT inputs, 16-byte loads)
    for (int it = tid; it < EXT * (PT / 4); it += 256) {
      const int yy = it >> 3, x0 = (it & 7) * 4;
      float wv[NT + 3 + 3];                                                     // rounded up to whole float4s
      constexpr int NV = (NT + 3 + 3) / 4;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const float4 q = *reinterpret_cast<const float4*>(&s_in[yy][x0 + 4 * v]);
        wv[4 * v] = q.x; wv[4 * v + 1] = q.y; wv[4 * v + 2] = q.z; wv[4 * v + 3] = q.w;
      }
      float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int t = 0; t < NT; ++t) {
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = fmaf(tp[t], wv[t + j], a[j]);
      }
      *reinterpret_cast<float4*>(&s_h[yy][x0]) = make_float4(a[0], a[1], a[2], a[3]);
    }
    __syncthreads();
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const float4 q = *reinterpret_cast<const float4*>(&s_h[ly + t][lx]);
      v[0] = fmaf(tp[t], q.x, v[0]); v[1] = fmaf(tp[t], q.y, v[1]); v[2] = fmaf(tp[t], q.z, v[2]); v[3] = fmaf(tp[t], q.w, v[3]);
    }
    if (eps != 0.f && oy < H) {
      const int64_t e0 = ((int64_t)c * H + oy) * W + ox;   // element index inside the sample
      float z[4];
      if (noise != nullptr) {
#pragma unroll
        for (int j = 0; j < 4; ++j) z[j] = (ox + j < W) ? __ldg(noise + (int64_t)b * C * H * W + e0 + j) : 0.f;
      } else {
        if ((e0 & 3) == 0) {
          philox_normal4(seed, noise_stream(sample0 + b, 0), (uint64_t)(e0 >> 2), z);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) z[j] = philox_normal(seed, noise_stream(sample0 + b, 0), (uint64_t)(e0 + j));
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = fmaf(z[j], scale, v[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float r = fminf(fmaxf(v[j], 0.f), 1.f);
      if (pre != nullptr && oy < H && ox + j < W) pre[(((int64_t)b * C + c) * H + oy) * W + ox + j] = v[j];   // saved UNCLAMPED
      res[c][j] = normalize ? (r - 0.5f) * 2.0f : r;
    }
  }
  if (oy < H) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (ox + j >= W) continue;
      const int64_t o = (((int64_t)b * H + oy) * W + ox + j) * C;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < C) st1d(out, out_dtype, o + c, res[c][j]);
    }
  }
}


// ============================================================================ whole-image pre-processing (3 x 64 x 64: the `ids` configs)
// One CTA per image: the image (48 KB) lives in shared memory for the whole kernel -- ONE read of x from HBM, ONE write of the result.
// The N(0,1) noise is drawn once (Philox, same stream and counters as the tiled kernels above, or read from the explicit tensor), kept in
// registers while its L2 norm is reduced inside the CTA (fixed order: bit-reproducible), and added after the blur: no separate
// sum-of-squares kernel, no second Philox pass.  Blur = separable 15-tap Gaussian with reflect border (abstract_models.py:145-159):
// horizontal pass from a row layout with the reflected halo materialised (16-byte window loads), vertical pass register-blocked over 8
// output rows (22 row loads for 8 output quads instead of 15 per quad).  Replaces preprocess_blur_fast_kernel<7> / preprocess_fwd_kernel
// + noise_sumsq_* at this size (they ran at 5-16% of the HBM roofline: two Philox passes, 4 re-staged tiles per image and channel).
constexpr int PI_HW = 64, PI_C = 3, PI_PITCH = 80, PI_OFF = 8;      // row = [8 halo | 64 data | 8 halo] floats
constexpr int PI_SMEM_BYTES = (PI_C * PI_HW * PI_PITCH + PI_C * PI_HW * PI_HW) * 4;

template <int RT>
__global__ void __launch_bounds__(256, 2) preprocess_image_kernel(const float* __restrict__ x, const float* __restrict__ noise, SeedArg seed_arg,
                                                                   int64_t sample0, float eps, const float* __restrict__ taps, int normalize,
                                                                   void* out, int out_dtype, float* __restrict__ pre) {
  extern __shared__ __align__(16) float pi_smem[];
  float* s_x = pi_smem;                                    // [3][64][80]; re-used as s_v [3][64][64] after the horizontal pass
  float* s_h = pi_smem + PI_C * PI_HW * PI_PITCH;          // [3][64][64]
  constexpr int HW = PI_HW * PI_HW, CHW = PI_C * HW;
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* xb = x + (int64_t)b * CHW;
  // ---- image -> shared memory (data columns at offset 8: 16-byte aligned)
#pragma unroll
  for (int k = 0; k < CHW / 4 / 256; ++k) {
    const int q = tid + k * 256;
    const int c = q / (HW / 4), r = q - c * (HW / 4), y = r >> 4, xq = r & 15;
    const float4 v = __ldg(reinterpret_cast<const float4*>(xb) + q);
    *reinterpret_cast<float4*>(&s_x[(c * PI_HW + y) * PI_PITCH + PI_OFF + 4 * xq]) = v;
  }
  // ---- noise of this thread's output items (item = 4 pixels x 3 channels), norm reduced in the CTA
  float z[4][PI_C][4];
  float scale = 0.f;
  if (eps != 0.f) {
    const uint64_t seed = seed_arg.get();
    const uint64_t stream = noise_stream(sample0 + b, 0);
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int it = tid + k * 256, y = it >> 4, xq = it & 15;
#pragma unroll
      for (int c = 0; c < PI_C; ++c) {
        const int e4 = ((c * PI_HW + y) * PI_HW + 4 * xq) >> 2;
        if (noise != nullptr) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(noise + (int64_t)b * CHW) + e4);
          z[k][c][0] = v.x; z[k][c][1] = v.y; z[k][c][2] = v.z; z[k][c][3] = v.w;
        } else {
          philox_normal4(seed, stream, (uint64_t)e4, z[k][c]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) acc = fmaf(z[k][c][j], z[k][c][j], acc);
      }
    }
    scale = eps / sqrtf(block_sum_256(acc));
  }
  __syncthreads();
  const float* s_v = s_x + PI_OFF;                         // un-blurred: read the data columns in place (pitch 80)
  int v_pitch = PI_PITCH;
  if (RT > 0) {
    float tp[2 * RT + 1];
#pragma unroll
    for (int t = 0; t < 2 * RT + 1; ++t) tp[t] = __ldg(taps + t);
    // ---- reflected halo columns: x = -k -> k, x = 63 + k -> 63 - k
    for (int i = tid; i < PI_C * PI_HW * 2 * RT; i += 256) {
      const int row = i / (2 * RT), k = i - row * (2 * RT);
      float* rp = s_x + row * PI_PITCH + PI_OFF;
      if (k < RT) rp[-(k + 1)] = rp[k + 1];
      else rp[PI_HW + (k - RT)] = rp[PI_HW - 2 - (k - RT)];
    }
    __syncthreads();
    // ---- horizontal pass: item = 4 consecutive outputs of one row
#pragma unroll 1
    for (int k = 0; k < CHW / 4 / 256; ++k) {
      const int q = tid + k * 256;
      const int row = q >> 4, xq = q & 15;
      const float* rp = s_x + row * PI_PITCH + 4 * xq;     // window: columns (4 xq + 8 - RT) .. (4 xq + 11 + RT) of the padded row
      constexpr int W0 = PI_OFF - RT;                      // first needed column relative to rp
      constexpr int NV = (W0 + 2 * RT + 4 + 3) / 4;
      float wv[4 * NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const float4 t4 = *reinterpret_cast<const float4*>(rp + 4 * v);
        wv[4 * v] = t4.x; wv[4 * v + 1] = t4.y; wv[4 * v + 2] = t4.z; wv[4 * v + 3] = t4.w;
      }
      float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int t = 0; t < 2 * RT + 1; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = fmaf(tp[t], wv[W0 + t + j], a[j]);
      *reinterpret_cast<float4*>(&s_h[row * PI_HW + 4 * xq]) = make_float4(a[0], a[1], a[2], a[3]);
    }
    __syncthreads();
    // ---- vertical pass: item = (channel, 4-pixel column, block of 8 rows); results over the (now free) s_x region, pitch 64
    float* s_o = s_x;
    for (int it = tid; it < PI_C * 16 * 8; it += 256) {
      const int c = it >> 7, r = it & 127, yb = r >> 4, xq = r & 15;
      const float* cp = s_h + c * HW + 4 * xq;
      float a[8][4];
#pragma unroll
      for (int o = 0; o < 8; ++o) { a[o][0] = 0.f; a[o][1] = 0.f; a[o][2] = 0.f; a[o][3] = 0.f; }
#pragma unroll
      for (int i = 0; i < 8 + 2 * RT; ++i) {
        const int yy = reflect_idx(yb * 8 + i - RT, PI_HW);
        const float4 t4 = *reinterpret_cast<const float4*>(cp + yy * PI_HW);
#pragma unroll
        for (int o = 0; o < 8; ++o) {
          const int t = i - o;                             // input row i feeds output row o through tap t
          if (t < 0 || t > 2 * RT) continue;
          a[o][0] = fmaf(tp[t], t4.x, a[o][0]); a[o][1] = fmaf(tp[t], t4.y, a[o][1]);
          a[o][2] = fmaf(tp[t], t4.z, a[o][2]); a[o][3] = fmaf(tp[t], t4.w, a[o][3]);
        }
      }
#pragma unroll
      for (int o = 0; o < 8; ++o)
        *reinterpret_cast<float4*>(&s_o[(c * PI_HW + yb * 8 + o) * PI_HW + 4 * xq]) = make_float4(a[o][0], a[o][1], a[o][2], a[o][3]);
    }
    __syncthreads();
    s_v = s_x;
    v_pitch = PI_HW;
  }
  // ---- + noise, clamp, normalise; NHWC out: the 12 values of an item are contiguous
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int it = tid + k * 256, y = it >> 4, xq = it & 15;
    float res[PI_C][4];
#pragma unroll
    for (int c = 0; c < PI_C; ++c) {
      const float4 t4 = *reinterpret_cast<const float4*>(s_v + (c * PI_HW + y) * v_pitch + 4 * xq);
      float v[4] = {t4.x, t4.y, t4.z, t4.w};
      if (eps != 0.f) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = fmaf(z[k][c][j], scale, v[j]);
      }
      if (pre != nullptr)    // saved UNCLAMPED (clamp backward mask)
        *reinterpret_cast<float4*>(pre + (int64_t)b * CHW + (c * PI_HW + y) * PI_HW + 4 * xq) = make_float4(v[0], v[1], v[2], v[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float r = fminf(fmaxf(v[j], 0.f), 1.f);
        res[c][j] = normalize ? (r - 0.5f) * 2.0f : r;
      }
    }
    const int64_t o = ((int64_t)b * HW + y * PI_HW + 4 * xq) * PI_C;
    if (out_dtype == GA_F32) {
      float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + o);
      op[0] = make_float4(res[0][0], res[1][0], res[2][0], res[0][1]);
      op[1] = make_float4(res[1][1], res[2][1], res[0][2], res[1][2]);
      op[2] = make_float4(res[2][2], res[0][3], res[1][3], res[2][3]);
    } else {
      uint2* op = reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + o);
      op[0] = make_uint2(pack_bf16x2(res[0][0], res[1][0]), pack_bf16x2(res[2][0], res[0][1]));
      op[1] = make_uint2(pack_bf16x2(res[1][1], res[2][1]), pack_bf16x2(res[0][2], res[1][2]));
      op[2] = make_uint2(pack_bf16x2(res[2][2], res[0][3]), pack_bf16x2(res[1][3], res[2][3]));
    }
  }
}

// backward helpers: g (NHWC) -> masked/scaled NCHW;  1-D transposed reflect-border blur along one axis
__global__ void preprocess_bwd_mask_kernel(const void* __restrict__ g, int g_dtype, const float* __restrict__ pre,
                                           float gscale, int C, int H, int W, int64_t total, float* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int x = (int)(i % W); int64_t t = i / W;
  int y = (int)(t % H); t /= H;
  int c = (int)(t % C); int64_t b = t / C;
  float p = pre[i];
  float gv = ld1d(g, g_dtype, ((b * H + y) * W + x) * C + c);
  out[i] = (p >= 0.f && p <= 1.f) ? gv * gscale : 0.f;
}

__global__ void blur_transpose_1d_kernel(const float* __restrict__ in, const float* __restrict__ taps, int R, int H, int W,
                                         int axis /*0 = y, 1 = x*/, int64_t total, float* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int x = (int)(i % W);
  const int y = (int)((i / W) % H);
  const int64_t plane = i / ((int64_t)H * W) * H * W;
  const int n = axis == 0 ? H : W;
  const int pos = axis == 0 ? y : x;
  const int64_t stride = axis == 0 ? W : 1;
  const float* base = in + plane + (axis == 0 ? x : (int64_t)y * W);
  float acc = 0.f;
  for (int d = -R; d <= R; ++d) {
    const float w = taps[d + R];
    int j = pos - d;                         // direct: j + d = pos
    if (j >= 0 && j < n) acc = fmaf(w, base[j * stride], acc);
    if (pos > 0) {                           // left reflection: j + d = -pos
      j = -pos - d;
      if (j >= 0 && j < n) acc = fmaf(w, base[j * stride], acc);
    }
    if (pos < n - 1) {                       // right reflection: j + d = 2n-2-pos
      j = 2 * n - 2 - pos - d;
      if (j >= 0 && j < n) acc = fmaf(w, base[j * stride], acc);
    }
  }
  out[i] = acc;
}

// ============================================================================ SE: channel sums + gate + residual
// partial[n][blk][c] = sum over the block's pixel slice (no atomics: bit-reproducible)
__global__ void __launch_bounds__(256) channel_sum_kernel(const void* __restrict__ r, int dtype, int HW, int C,
                                                          int pix_per_block, float* __restrict__ partial) {
  __shared__ float s_part[256];
  const int n = blockIdx.y;
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(p0 + pix_per_block, HW);
  const int64_t base = ((int64_t)n * HW + p0) * C;
  const int cnt = (p1 - p0) * C;
  float* dst = partial + ((int64_t)n * gridDim.x + blockIdx.x) * C;
  if (256 % C == 0) {          // each thread always sees the same channel (coalesced); a 4-channel vector variant measured slower
    float acc = 0.f;
    for (int i = threadIdx.x; i < cnt; i += 256) acc += ld1d(r, dtype, base + i);
    s_part[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < C) {
      float t = 0.f;
      for (int k = threadIdx.x; k < 256; k += C) t += s_part[k];
      dst[threadIdx.x] = t;
    }
  } else if (C % 256 == 0) {   // thread sees channels t, t+256, ... (coalesced)
    const int per = C / 256;
    for (int k = 0; k < per; ++k) {
      float acc = 0.f;
      for (int i = threadIdx.x + k * 256; i < cnt; i += C) acc += ld1d(r, dtype, base + i);
      dst[threadIdx.x + k * 256] = acc;
    }
  } else {                     // odd channel counts (tiny test architectures): one thread per channel
    for (int c = threadIdx.x; c < C; c += 256) {
      float acc = 0.f;
      for (int i = c; i < cnt; i += C) acc += ld1d(r, dtype, base + i);
      dst[c] = acc;
    }
  }
}

struct SeParams {
  const void* r; int r_dtype;
  const float* sums; const float* w1; const float* b1; const float* w2; const float* b2;
  int hidden; float res_scale;
  const void* skip; int skip_dtype;
  void* out; int out_dtype;
  void* out2; int out2_dtype;
  void* act; int act_dtype; const float* act_scale; const float* act_shift; int act_op;
  float* gate_out;
  int HW, C, pix_per_block, nparts;
  int act_rtf;                 // round the fp32 `act` copy to TF32 (it feeds a kind::tf32 conv)
};

__global__ void __launch_bounds__(256) se_residual_kernel(SeParams p) {
  extern __shared__ float sm[];      // mean[C] | gate[C] | hid[hidden]
  float* s_mean = sm;
  float* s_gate = sm + p.C;
  float* s_hid = sm + 2 * p.C;
  const int n = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float inv = 1.0f / (float)p.HW;
  for (int c = tid; c < p.C; c += 256) {
    float t = 0.f;
    for (int k = 0; k < p.nparts; ++k) t += p.sums[((int64_t)n * p.nparts + k) * p.C + c];   // fixed order
    s_mean[c] = t * inv;
  }
  __syncthreads();
  for (int j = warp; j < p.hidden; j += 8) {
    float a = 0.f;
    for (int c = lane; c < p.C; c += 32) a = fmaf(p.w1[(int64_t)j * p.C + c], s_mean[c], a);
    a = warp_sum(a);
    if (lane == 0) s_hid[j] = fmaxf(a + (p.b1 != nullptr ? p.b1[j] : 0.f), 0.f);
  }
  __syncthreads();
  for (int c = tid; c < p.C; c += 256) {
    float a = p.b2 != nullptr ? p.b2[c] : 0.f;
    for (int j = 0; j < p.hidden; ++j) a = fmaf(p.w2[(int64_t)c * p.hidden + j], s_hid[j], a);
    float g = sigmoidf_(a);
    s_gate[c] = g;
    if (p.gate_out != nullptr && blockIdx.x == 0) p.gate_out[(int64_t)n * p.C + c] = g;
  }
  __syncthreads();
  const int p0 = blockIdx.x * p.pix_per_block;
  const int p1 = min(p0 + p.pix_per_block, p.HW);
  const int c4n = p.C >> 2;
  const int64_t base = ((int64_t)n * p.HW + p0) * p.C;
  const int cnt4 = (p1 - p0) * c4n;
  // 4 independent vector items per thread per trip: all loads are issued before the first store (the output may alias
  // nothing, but the compiler cannot know; a rolled loop kept ONE load pair in flight per thread)
  for (int i0 = tid; i0 < cnt4; i0 += 256 * 4) {
    float rv[4][4], sv[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 256;
      if (i < cnt4) {
        const int64_t off = base + (int64_t)i * 4;
        ld4d(p.r, p.r_dtype, off, rv[u]);
        ld4d(p.skip, p.skip_dtype, off, sv[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 256;
      if (i >= cnt4) continue;
      const int c = (i % c4n) * 4;
      const int64_t off = base + (int64_t)i * 4;
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = fmaf(p.res_scale * s_gate[c + j], rv[u][j], sv[u][j]);
      st4d(p.out, p.out_dtype, off, o);
      if (p.out2 != nullptr) st4d(p.out2, p.out2_dtype, off, o);
      if (p.act != nullptr) {
        float a[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float t = p.act_scale != nullptr ? fmaf(o[j], p.act_scale[c + j], p.act_shift[c + j]) : o[j];
          a[j] = p.act_op == GA_ACT_SILU ? silu_fast(t) : (p.act_op == GA_ACT_ELU ? (t > 0.f ? t : __expf(t) - 1.0f) : t);
          if (p.act_rtf) a[j] = round_tf32(a[j]);
        }
        st4d(p.act, p.act_dtype, off, a);
      }
    }
  }
}

// ============================================================================ latent mix
// one thread per pixel: q / p / z rows are contiguous per pixel (vector-friendly, every byte of a line is used), the
// NCHW eps reads are coalesced across the warp (adjacent threads = adjacent pixels)
__global__ void __launch_bounds__(128) latent_mix_kernel(const void* __restrict__ q, int q_dtype, int Cq,
                                                         const void* __restrict__ pp, int p_dtype, const float* __restrict__ eps,
                                                         SeedArg seed_arg, int level, int64_t sample0,
                                                         const float* __restrict__ alpha_dev, float temp, int Z, int64_t total_pix,
                                                         int HW, void* __restrict__ zout, int z_dtype, int Cz) {
  const uint64_t seed = seed_arg.get();
  const int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= total_pix) return;
  const int64_t n = pix / HW;
  const int hw = (int)(pix % HW);
  const float a = *alpha_dev;
  const float* e_base = eps != nullptr ? eps + n * Z * HW + hw : nullptr;
  const uint64_t stream = noise_stream(sample0 + n, level + 1);
  const bool fast = false;     // (MUFU tanh / exp measured no faster once the loads were vectorised, and cost 5e-4 of the 1e-2 budget)
  for (int z0 = 0; z0 < Cz; z0 += 4) {             // 4 channels per trip: their loads are issued together
    float mq[4], mp[4], lp[4], ee[4];
    if (e_base == nullptr && z0 < Z) latent_eps4(seed, stream, z0 >> 2, hw, HW, ee);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int zc = z0 + u;
      mq[u] = mp[u] = lp[u] = 0.f;
      if (zc < Z) {
        mq[u] = ld1d(q, q_dtype, pix * Cq + zc);
        if (e_base != nullptr) ee[u] = __ldg(e_base + (int64_t)zc * HW);
        if (pp != nullptr) {
          mp[u] = ld1d(pp, p_dtype, pix * (2 * Z) + zc);
          lp[u] = ld1d(pp, p_dtype, pix * (2 * Z) + Z + zc);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int zc = z0 + u;
      if (zc >= Cz) continue;
      float out = 0.f;                             // channels >= Z: zero padding (tensor-core K padding)
      if (zc < Z) {
        if (fast) {
          if (pp == nullptr) out = (1.f - a) * (5.f * tanh_approx(0.2f * mq[u])) + a * (ee[u] * temp);
          else out = (1.f - a) * (5.f * tanh_approx(0.2f * (mp[u] + mq[u]))) +
                     a * (5.f * tanh_approx(0.2f * mp[u]) + ee[u] * (temp * __expf(5.f * tanh_approx(0.2f * lp[u]))));
        } else {
          if (pp == nullptr) out = (1.f - a) * softclamp5_(mq[u]) + a * (ee[u] * temp);
          else out = latent_mix_prior(a, mq[u], mp[u], lp[u], ee[u], temp);
        }
      }
      st1d(zout, z_dtype, pix * Cz + zc, out);
    }
  }
}

// vectorised variant (Z, Cq, Cz multiples of 4): one thread per (pixel, 4-channel group), adjacent threads = adjacent 16-byte pieces of
// the pixel rows, so every load / store instruction of a warp covers whole 128-byte lines (the per-pixel kernel above issues 60
// scalar loads whose 32 lanes hit 32 different lines: L1 wavefront bound, 5x slower at 32x32)
__global__ void __launch_bounds__(256) latent_mix_vec4_kernel(const void* __restrict__ q, int q_dtype, int Cq, const void* __restrict__ pp,
                                                              int p_dtype, const float* __restrict__ eps, SeedArg seed_arg, int level,
                                                              int64_t sample0, const float* __restrict__ alpha_dev, float temp, int Z,
                                                              int64_t total_pix, int HW, void* __restrict__ zout, int z_dtype, int Cz) {
  const uint64_t seed = seed_arg.get();
  const int groups = Cz >> 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total_pix * groups) return;
  const int j = (int)(idx % groups);
  const int64_t pix = idx / groups;
  float out[4] = {0.f, 0.f, 0.f, 0.f};               // channel groups >= Z: zero padding (tensor-core K padding)
  if (4 * j < Z) {
    const int64_t n = pix / HW;
    const int hw = (int)(pix % HW);
    const float a = *alpha_dev;
    float mq[4], mp[4] = {0.f, 0.f, 0.f, 0.f}, lp[4] = {0.f, 0.f, 0.f, 0.f}, ee[4];
    ld4d(q, q_dtype, pix * Cq + 4 * j, mq);
    if (pp != nullptr) {
      ld4d(pp, p_dtype, pix * (2 * Z) + 4 * j, mp);
      ld4d(pp, p_dtype, pix * (2 * Z) + Z + 4 * j, lp);
    }
    if (eps != nullptr) {
#pragma unroll
      for (int u = 0; u < 4; ++u) ee[u] = __ldg(eps + (n * Z + 4 * j + u) * HW + hw);
    } else {
      latent_eps4(seed, noise_stream(sample0 + n, level + 1), j, hw, HW, ee);
    }
    const bool fast = false;   // see latent_mix_kernel
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (fast) {
        if (pp == nullptr) out[u] = (1.f - a) * (5.f * tanh_approx(0.2f * mq[u])) + a * (ee[u] * temp);
        else out[u] = (1.f - a) * (5.f * tanh_approx(0.2f * (mp[u] + mq[u]))) +
                      a * (5.f * tanh_approx(0.2f * mp[u]) + ee[u] * (temp * __expf(5.f * tanh_approx(0.2f * lp[u]))));
      } else {
        if (pp == nullptr) out[u] = (1.f - a) * softclamp5_(mq[u]) + a * (ee[u] * temp);
        else out[u] = latent_mix_prior(a, mq[u], mp[u], lp[u], ee[u], temp);
      }
    }
  }
  st4d(zout, z_dtype, pix * Cz + 4 * j, out);
}

// ============================================================================ DiscMixLogistic mean
constexpr int DM_PIX = 128;          // one pixel per thread
__global__ void __launch_bounds__(128) discmix_mean_kernel(const void* __restrict__ logits, int dtype, int n_mix, int HW,
                                                           int64_t total_pix, float* __restrict__ purified, void* cls,
                                                           int cls_dtype) {
  extern __shared__ float s_l[];   // [DM_PIX][CL + 1]
  const int CL = 10 * n_mix;
  const int pitch = CL + 1;
  const int64_t pix0 = (int64_t)blockIdx.x * DM_PIX;
  const int npx = (int)min((int64_t)DM_PIX, total_pix - pix0);
  const int cnt = npx * CL;
  // element i = tid + 128 k of the tile goes to row i / CL, column i % CL: tracked incrementally (a division per element was ~2/3 of
  // this kernel's instructions)
  const int dp = 128 / CL, dc = 128 % CL;
  int rp = threadIdx.x / CL, rc = threadIdx.x % CL;
  for (int i0 = threadIdx.x; i0 < cnt; i0 += 128 * 8) {          // 8 loads in flight per thread
    float t[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * 128;
      t[u] = i < cnt ? ld1d(logits, dtype, pix0 * CL + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * 128;
      if (i < cnt) s_l[rp * pitch + rc] = t[u];
      rp += dp; rc += dc;
      if (rc >= CL) { rc -= CL; ++rp; }
    }
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t >= npx) return;
  const float* l = s_l + t * pitch;
  float mx = l[0];
  for (int m = 1; m < n_mix; ++m) mx = fmaxf(mx, l[m]);
  float den = 0.f, mu0 = 0.f, mu1 = 0.f, mu2 = 0.f, k0 = 0.f, k1 = 0.f, k2 = 0.f;
  for (int m = 0; m < n_mix; ++m) {
    const float e = expf(l[m] - mx);
    const float* q = l + n_mix + 9 * m;   // [m0 m1 m2 | s0 s1 s2 | k0 k1 k2]
    den += e;
    mu0 = fmaf(e, q[0], mu0); mu1 = fmaf(e, q[1], mu1); mu2 = fmaf(e, q[2], mu2);
    k0 = fmaf(e, tanhf(q[6]), k0); k1 = fmaf(e, tanhf(q[7]), k1); k2 = fmaf(e, tanhf(q[8]), k2);
  }
  const float inv = 1.f / den;
  mu0 *= inv; mu1 *= inv; mu2 *= inv; k0 *= inv; k1 *= inv; k2 *= inv;
  const float r = fminf(fmaxf(mu0, -1.f), 1.f);
  const float g = fminf(fmaxf(fmaf(k0, r, mu1), -1.f), 1.f);
  const float b = fminf(fmaxf(mu2 + k1 * r + k2 * g, -1.f), 1.f);
  const int64_t pix = pix0 + t;
  const int64_t n = pix / HW, hw = pix % HW;
  float* dst = purified + n * 3 * HW + hw;
  dst[0] = r * 0.5f + 0.5f; dst[HW] = g * 0.5f + 0.5f; dst[2 * (int64_t)HW] = b * 0.5f + 0.5f;
  if (cls != nullptr) {
    // classifier input normalize(purified, 0.5, 0.5) (abstract_models.py:60)
    st1d(cls, cls_dtype, pix * 3 + 0, ((r * 0.5f + 0.5f) - 0.5f) * 2.0f);
    st1d(cls, cls_dtype, pix * 3 + 1, ((g * 0.5f + 0.5f) - 0.5f) * 2.0f);
    st1d(cls, cls_dtype, pix * 3 + 2, ((b * 0.5f + 0.5f) - 0.5f) * 2.0f);
  }
}

// ============================================================================ resampling / layout
__global__ void upsample_nearest2x_kernel(const void* in, int in_dtype, void* out, int out_dtype, int N, int H, int W, int C) {
  const int c4n = C >> 2;
  const int Ho = 2 * H, Wo = 2 * W;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * c4n) return;
  const int c = (int)(idx % c4n) * 4;
  int64_t t = idx / c4n;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  float v[4];
  ld4d(in, in_dtype, ((n * H + (y >> 1)) * W + (x >> 1)) * C + c, v);
  st4d(out, out_dtype, ((n * Ho + y) * Wo + x) * C + c, v);
}

__global__ void upsample_bilinear2x_kernel(const void* in, int in_dtype, void* out, int out_dtype, int N, int H, int W, int C) {
  const int c4n = C >> 2;
  const int Ho = 2 * H, Wo = 2 * W;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * c4n) return;
  const int c = (int)(idx % c4n) * 4;
  int64_t t = idx / c4n;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  // align_corners=True: src = dst * (in-1)/(out-1)
  const float sy = Ho > 1 ? (float)(H - 1) / (float)(Ho - 1) : 0.f;
  const float sx = Wo > 1 ? (float)(W - 1) / (float)(Wo - 1) : 0.f;
  const float fy = sy * y, fx = sx * x;
  int y0 = (int)fy, x0 = (int)fx;
  y0 = min(y0, H - 1); x0 = min(x0, W - 1);
  const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
  const float wy = fy - y0, wx = fx - x0;
  float a[4], b[4], cc[4], d[4], o[4];
  ld4d(in, in_dtype, ((n * H + y0) * W + x0) * C + c, a);
  ld4d(in, in_dtype, ((n * H + y0) * W + x1) * C + c, b);
  ld4d(in, in_dtype, ((n * H + y1) * W + x0) * C + c, cc);
  ld4d(in, in_dtype, ((n * H + y1) * W + x1) * C + c, d);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float top = a[j] + wx * (b[j] - a[j]);
    const float bot = cc[j] + wx * (d[j] - cc[j]);
    o[j] = top + wy * (bot - top);
  }
  st4d(out, out_dtype, ((n * Ho + y) * Wo + x) * C + c, o);
}

__global__ void maxpool2x2_kernel(const void* in, int in_dtype, void* out, int out_dtype, int N, int H, int W, int C) {
  const int c4n = C >> 2;
  const int Ho = H >> 1, Wo = W >> 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * c4n) return;
  const int c = (int)(idx % c4n) * 4;
  int64_t t = idx / c4n;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  float a[4], b[4], cc[4], d[4], o[4];
  const int64_t base = ((n * H + 2 * y) * W + 2 * x) * C + c;
  ld4d(in, in_dtype, base, a);
  ld4d(in, in_dtype, base + C, b);
  ld4d(in, in_dtype, base + (int64_t)W * C, cc);
  ld4d(in, in_dtype, base + (int64_t)W * C + C, d);
#pragma unroll
  for (int j = 0; j < 4; ++j) o[j] = fmaxf(fmaxf(a[j], b[j]), fmaxf(cc[j], d[j]));
  st4d(out, out_dtype, ((n * Ho + y) * Wo + x) * C + c, o);
}

// x[:, ::2, ::2, :]  (nn.MaxPool2d(1, 2) shortcut of the IR-SE50 bottlenecks, encoding/helpers.py:95-96)
__global__ void subsample2x_kernel(const void* in, int in_dtype, void* out, int out_dtype, int N, int H, int W, int C) {
  const int c4n = C >> 2;
  const int Ho = (H + 1) >> 1, Wo = (W + 1) >> 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * c4n) return;
  const int c = (int)(idx % c4n) * 4;
  int64_t t = idx / c4n;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  float v[4];
  ld4d(in, in_dtype, ((n * H + 2 * y) * W + 2 * x) * C + c, v);
  st4d(out, out_dtype, ((n * Ho + y) * Wo + x) * C + c, v);
}

// 3x3 max-pool, stride 2, pad 1 (torchvision ResNet stem)
__global__ void maxpool3x3s2_kernel(const void* in, int in_dtype, void* out, int out_dtype, int N, int H, int W, int C) {
  const int c4n = C >> 2;
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * c4n) return;
  const int c = (int)(idx % c4n) * 4;
  int64_t t = idx / c4n;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  for (int dy = -1; dy <= 1; ++dy) {
    const int iy = 2 * y + dy;
    if (iy < 0 || iy >= H) continue;
    for (int dx = -1; dx <= 1; ++dx) {
      const int ix = 2 * x + dx;
      if (ix < 0 || ix >= W) continue;
      float v[4];
      ld4d(in, in_dtype, ((n * H + iy) * W + ix) * C + c, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) m[j] = fmaxf(m[j], v[j]);
    }
  }
  st4d(out, out_dtype, ((n * Ho + y) * Wo + x) * C + c, m);
}

// global average pool: one block per image, fixed summation order (deterministic)
__global__ void __launch_bounds__(256) global_avgpool_kernel(const void* in, int in_dtype, int HW, int C, void* out, int out_dtype) {
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += 256) {
    float acc = 0.f;
    for (int p = 0; p < HW; ++p) acc += ld1d(in, in_dtype, ((int64_t)n * HW + p) * C + c);
    st1d(out, out_dtype, (int64_t)n * C + c, acc / (float)HW);
  }
}

__global__ void affine_act_kernel(const void* in, int in_dtype, const float* __restrict__ scale, const float* __restrict__ shift,
                                  int act, void* out, int out_dtype, int C, int64_t total, int rtf) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  float v = ld1d(in, in_dtype, idx);
  const int c = (int)(idx % C);
  if (scale != nullptr) v = fmaf(v, scale[c], shift[c]);
  v = apply_act(v, act);
  st1d(out, out_dtype, idx, rtf ? round_tf32(v) : v);
}

// 8 elements per thread (C % 8 == 0): 16/32-byte vector accesses
__global__ void __launch_bounds__(256) affine_act_vec8_kernel(const void* in, int in_dtype, const float* __restrict__ scale,
                                                              const float* __restrict__ shift, int act, void* out, int out_dtype,
                                                              int C, int64_t total8, int rtf) {
  int64_t i8 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i8 >= total8) return;
  const int64_t idx = i8 * 8;
  const int c = (int)(idx % C);
  float a[4], b[4];
  ld4d(in, in_dtype, idx, a);
  ld4d(in, in_dtype, idx + 4, b);
  if (scale != nullptr) {
    const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale + c)), s1 = __ldg(reinterpret_cast<const float4*>(scale + c + 4));
    const float4 h0 = __ldg(reinterpret_cast<const float4*>(shift + c)), h1 = __ldg(reinterpret_cast<const float4*>(shift + c + 4));
    a[0] = fmaf(a[0], s0.x, h0.x); a[1] = fmaf(a[1], s0.y, h0.y); a[2] = fmaf(a[2], s0.z, h0.z); a[3] = fmaf(a[3], s0.w, h0.w);
    b[0] = fmaf(b[0], s1.x, h1.x); b[1] = fmaf(b[1], s1.y, h1.y); b[2] = fmaf(b[2], s1.z, h1.z); b[3] = fmaf(b[3], s1.w, h1.w);
  }
  apply_act_n<4>(a, act);
  apply_act_n<4>(b, act);
  if (rtf) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { a[j] = round_tf32(a[j]); b[j] = round_tf32(b[j]); }
  }
  st4d(out, out_dtype, idx, a);
  st4d(out, out_dtype, idx + 4, b);
}

__global__ void nchw_to_nhwc_kernel(const float* __restrict__ in, void* out, int out_dtype, float scale, float shift, int N,
                                    int C, int H, int W) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over NHWC output
  if (idx >= (int64_t)N * C * H * W) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int x = (int)(t % W); t /= W;
  const int y = (int)(t % H);
  const int64_t n = t / H;
  st1d(out, out_dtype, idx, fmaf(in[((n * C + c) * H + y) * W + x], scale, shift));
}

// ============================================================================ attack inner loop
__global__ void pgd_linf_step_kernel(float* __restrict__ x_adv, const float* __restrict__ grad, const float* __restrict__ x_nat,
                                     float step, float eps, int64_t n4, int64_t numel) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) {
    float4 a = reinterpret_cast<float4*>(x_adv)[i];
    const float4 g = __ldg(reinterpret_cast<const float4*>(grad) + i);
    const float4 x = __ldg(reinterpret_cast<const float4*>(x_nat) + i);
    auto upd = [&](float av, float gv, float xv) {
      const float sg = (gv > 0.f) ? 1.f : ((gv < 0.f) ? -1.f : 0.f);
      float v = fmaf(step, sg, av);
      v = fminf(fmaxf(v, xv - eps), xv + eps);
      return fminf(fmaxf(v, 0.f), 1.f);
    };
    a.x = upd(a.x, g.x, x.x); a.y = upd(a.y, g.y, x.y); a.z = upd(a.z, g.z, x.z); a.w = upd(a.w, g.w, x.w);
    reinterpret_cast<float4*>(x_adv)[i] = a;
  }
  if (i == 0) {
    for (int64_t k = n4 * 4; k < numel; ++k) {
      const float gv = grad[k];
      const float sg = (gv > 0.f) ? 1.f : ((gv < 0.f) ? -1.f : 0.f);
      float v = fmaf(step, sg, x_adv[k]);
      v = fminf(fmaxf(v, x_nat[k] - eps), x_nat[k] + eps);
      x_adv[k] = fminf(fmaxf(v, 0.f), 1.f);
    }
  }
}

// one warp per sample
__global__ void softmax_xent_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels, int n, int classes,
                                    float* __restrict__ loss, float* __restrict__ dlogits, int32_t* __restrict__ pred,
                                    unsigned long long* __restrict__ n_correct) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const float* l = logits + (int64_t)warp * classes;
  float mx = -INFINITY; int arg = 0;
  for (int c = lane; c < classes; c += 32) {
    float v = l[c];
    if (v > mx) { mx = v; arg = c; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    float om = __shfl_xor_sync(0xffffffffu, mx, o);
    int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }   // first max wins, like torch.argmax
  }
  float den = 0.f;
  for (int c = lane; c < classes; c += 32) den += expf(l[c] - mx);
  den = warp_sum(den);
  const int64_t y = labels ? labels[warp] : -1;
  if (dlogits != nullptr) {
    const float invn = 1.f / (float)n;
    for (int c = lane; c < classes; c += 32) {
      float pr = expf(l[c] - mx) / den;
      dlogits[(int64_t)warp * classes + c] = (pr - (c == y ? 1.f : 0.f)) * invn;
    }
  }
  if (lane == 0) {
    if (loss != nullptr) loss[warp] = (y >= 0 && y < classes) ? logf(den) + mx - l[y] : 0.f;   // out-of-range label: no read past the row
    if (pred != nullptr) pred[warp] = arg;
    if (n_correct != nullptr && y >= 0 && arg == (int)y) atomicAdd(n_correct, 1ull);
  }
}

}  // namespace ga

// ================================================================================================ C ABI
using namespace ga;

extern "C" int ga_noise_sumsq_parts(int chw) { return max(1, min(GA_NOISE_PARTS, cdiv((chw + 3) / 4, 256))); }

extern "C" int ga_noise_sumsq(const float* noise, int n, int chw, float* sumsq, void* stream) {
  GA_CHECK(noise && sumsq && n >= 0 && chw > 0, "ga_noise_sumsq: bad arguments");
  if (n == 0) return 0;
  GA_CHECK((((uintptr_t)noise) & 15) == 0 && (chw % 4 == 0), "ga_noise_sumsq: noise must be 16-byte aligned with chw %% 4 == 0");
  noise_sumsq_kernel<<<dim3(ga_noise_sumsq_parts(chw), n), 256, 0, (cudaStream_t)stream>>>(noise, chw, sumsq);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_noise_sumsq_philox(uint64_t seed, int64_t sample0, int n, int chw, float* sumsq, void* stream) {
  GA_CHECK(sumsq && n >= 0 && chw > 0, "ga_noise_sumsq_philox: bad arguments");
  if (n == 0) return 0;
  noise_sumsq_philox_kernel<<<dim3(ga_noise_sumsq_parts(chw), n), 256, 0, (cudaStream_t)stream>>>(make_seed(seed, (cudaStream_t)stream), sample0, chw, sumsq);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_preprocess_fwd(const float* x, const float* noise, const float* sumsq, uint64_t seed, int64_t sample0,
                                 float eps, const float* taps, int radius, int normalize, const ga_tensor* out, float* pre,
                                 void* stream) {
  GA_CHECK(x && out && out->data, "ga_preprocess_fwd: null argument");
  GA_CHECK(out->c >= 1 && out->c <= 4, "ga_preprocess_fwd: image channels must be <= 4 (got %d)", out->c);
  GA_CHECK(radius >= 0 && radius <= MAXR, "ga_preprocess_fwd: blur radius %d > %d", radius, MAXR);
  GA_CHECK(eps == 0.f || sumsq, "ga_preprocess_fwd: eps != 0 needs the noise sum of squares");
  GA_CHECK(taps == nullptr || (radius < out->h && radius < out->w), "ga_preprocess_fwd: reflect border needs radius < image size");
  if (out->n == 0) return 0;
  const int tiles = cdiv(out->h, PT) * cdiv(out->w, PT);
  const int nparts = ga_noise_sumsq_parts(out->c * out->h * out->w);
  dim3 grid(tiles, 1, out->n);
  cudaStream_t s = (cudaStream_t)stream;
  if (taps != nullptr && radius == 7)
    preprocess_blur_fast_kernel<7><<<grid, 256, 0, s>>>(x, noise, sumsq, make_seed(seed, (cudaStream_t)stream), nparts, sample0, eps, taps, normalize, out->c, out->h,
                                                       out->w, out->data, out->dtype, pre);
  else if (taps != nullptr && radius == 12)
    preprocess_blur_fast_kernel<12><<<grid, 256, 0, s>>>(x, noise, sumsq, make_seed(seed, (cudaStream_t)stream), nparts, sample0, eps, taps, normalize, out->c, out->h,
                                                        out->w, out->data, out->dtype, pre);
  else if (taps != nullptr)
    preprocess_fwd_kernel<true><<<grid, 256, 0, s>>>(x, noise, sumsq, make_seed(seed, (cudaStream_t)stream), nparts, sample0, eps, taps, radius, normalize, out->c,
                                                    out->h, out->w, out->data, out->dtype, pre);
  else
    preprocess_fwd_kernel<false><<<grid, 256, 0, s>>>(x, noise, sumsq, make_seed(seed, (cudaStream_t)stream), nparts, sample0, eps, nullptr, 0, normalize, out->c,
                                                     out->h, out->w, out->data, out->dtype, pre);
  GA_LAUNCH_OK();
  return 0;
}


extern "C" int ga_preprocess_image_supported(int c, int h, int w, int radius, int have_taps) {
  return (c == PI_C && h == PI_HW && w == PI_HW && (!have_taps || radius == 7)) ? 1 : 0;
}

// blur -> noise -> clamp -> normalise for 3 x 64 x 64 images in ONE launch (the noise norm is reduced inside the kernel: no sumsq pre-pass)
extern "C" int ga_preprocess_image_fwd(const float* x, const float* noise, uint64_t seed, int64_t sample0, float eps, const float* taps,
                                       int radius, int normalize, const ga_tensor* out, float* pre, void* stream) {
  GA_CHECK(x && out && out->data, "ga_preprocess_image_fwd: null argument");
  GA_CHECK(ga_preprocess_image_supported(out->c, out->h, out->w, radius, taps != nullptr), "ga_preprocess_image_fwd: unsupported shape");
  GA_CHECK(out->dtype == GA_F32 || out->dtype == GA_BF16, "ga_preprocess_image_fwd: out must be fp32 or bf16");
  if (out->n == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  static bool configured = false;
  if (!configured) {
    GA_CUDA(cudaFuncSetAttribute(preprocess_image_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, PI_SMEM_BYTES));
    GA_CUDA(cudaFuncSetAttribute(preprocess_image_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PI_SMEM_BYTES));
    configured = true;
  }
  if (taps != nullptr)
    preprocess_image_kernel<7><<<out->n, 256, PI_SMEM_BYTES, s>>>(x, noise, make_seed(seed, s), sample0, eps, taps, normalize, out->data, out->dtype, pre);
  else
    preprocess_image_kernel<0><<<out->n, 256, PI_SMEM_BYTES, s>>>(x, noise, make_seed(seed, s), sample0, eps, nullptr, normalize, out->data, out->dtype, pre);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_preprocess_bwd(const ga_tensor* g, const float* pre, const float* taps, int radius, int normalize,
                                 float* tmp, float* gx, void* stream) {
  GA_CHECK(g && pre && gx, "ga_preprocess_bwd: null argument");
  GA_CHECK(taps == nullptr || tmp != nullptr, "ga_preprocess_bwd: blur backward needs a workspace");
  const int64_t total = numel(g);
  if (total == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int blocks = cdiv(total, 256);
  preprocess_bwd_mask_kernel<<<blocks, 256, 0, s>>>(g->data, g->dtype, pre, normalize ? 2.0f : 1.0f, g->c, g->h, g->w, total, gx);
  GA_LAUNCH_OK();
  if (taps != nullptr) {
    blur_transpose_1d_kernel<<<blocks, 256, 0, s>>>(gx, taps, radius, g->h, g->w, 0, total, tmp);
    GA_LAUNCH_OK();
    blur_transpose_1d_kernel<<<blocks, 256, 0, s>>>(tmp, taps, radius, g->h, g->w, 1, total, gx);
    GA_LAUNCH_OK();
  }
  return 0;
}

static int se_pix_per_block(int HW, int n) {
  // fixed slice of 128 pixels, independent of the batch size: a sample's reduction order (hence its bits) does
  // not depend on how the batch is sharded over GPUs
  (void)n;
  return HW < 128 ? HW : 128;
}

extern "C" int ga_channel_sum_parts(int n, int hw) { return cdiv(hw, se_pix_per_block(hw, n)); }

extern "C" int ga_channel_sum(const ga_tensor* r, float* sums, void* stream) {
  GA_CHECK(r && sums, "ga_channel_sum: null argument");
  if (numel(r) == 0) return 0;
  const int HW = r->h * r->w;
  const int ppb = se_pix_per_block(HW, r->n);
  channel_sum_kernel<<<dim3(cdiv(HW, ppb), r->n), 256, 0, (cudaStream_t)stream>>>(r->data, r->dtype, HW, r->c, ppb, sums);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_se_residual_fwd(const ga_tensor* r, const float* sums, const float* w1, const float* b1, const float* w2,
                                  const float* b2, int hidden, float res_scale, const ga_tensor* skip, const ga_tensor* out,
                                  const ga_tensor* out2, const ga_tensor* act, const float* act_scale, const float* act_shift,
                                  int act_op, float* gate_out, void* stream) {
  GA_CHECK(r && sums && w1 && w2 && skip && out, "ga_se_residual_fwd: null argument");
  GA_CHECK(act_op == GA_ACT_SILU || act_op == GA_ACT_NONE || act_op == GA_ACT_ELU, "ga_se_residual_fwd: act_op must be SILU, ELU or NONE");
  GA_CHECK(same_shape(r, skip) && same_shape(r, out), "ga_se_residual_fwd: shape mismatch");
  GA_CHECK((r->c % 4) == 0, "ga_se_residual_fwd: channels must be a multiple of 4");
  GA_CHECK(!act || same_shape(r, act), "ga_se_residual_fwd: act output shape mismatch");
  GA_CHECK((act_scale == nullptr) == (act_shift == nullptr), "ga_se_residual_fwd: act_scale and act_shift go together");
  GA_CHECK(!out2 || same_shape(r, out2), "ga_se_residual_fwd: out2 shape mismatch");
  if (numel(r) == 0) return 0;
  SeParams p;
  p.r = r->data; p.r_dtype = r->dtype; p.sums = sums; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2;
  p.hidden = hidden; p.res_scale = res_scale;
  p.skip = skip->data; p.skip_dtype = skip->dtype;
  p.out = out->data; p.out_dtype = out->dtype;
  p.out2 = out2 ? out2->data : nullptr; p.out2_dtype = out2 ? out2->dtype : GA_F32;
  p.act = act ? act->data : nullptr; p.act_dtype = act ? act->dtype : GA_F32;
  p.act_scale = act_scale; p.act_shift = act_shift; p.act_op = act_op; p.gate_out = gate_out;
  p.act_rtf = (act && act->dtype == GA_F32 && round_tf32_enabled()) ? 1 : 0;
  p.HW = r->h * r->w; p.C = r->c;
  p.nparts = cdiv(p.HW, se_pix_per_block(p.HW, r->n));          // slicing of the channel sums: fixed 128 pixels
  // a CTA recomputes the gate MLP (three block-wide phases of dependent loads) before it streams: up to 512 pixels of an image per CTA so that
  // the preamble is paid 4x less often at 32x32
  static int apply_ppb_max = -1;
  if (apply_ppb_max < 0) { const char* e = getenv("GA_SE_APPLY_PPB"); apply_ppb_max = e ? atoi(e) : 512; }
  p.pix_per_block = p.HW < apply_ppb_max ? p.HW : apply_ppb_max;
  const size_t smem = (2 * (size_t)p.C + hidden) * sizeof(float);
  GA_CHECK(smem <= 48 * 1024, "ga_se_residual_fwd: too many channels");
  se_residual_kernel<<<dim3(cdiv(p.HW, p.pix_per_block), r->n), 256, smem, (cudaStream_t)stream>>>(p);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_latent_mix_fwd(const ga_tensor* q, const ga_tensor* p, const float* eps, uint64_t seed, int level,
                                 int64_t sample0, const float* alpha_dev, float temperature, int zdim, const ga_tensor* z,
                                 void* stream) {
  GA_CHECK(q && z && alpha_dev, "ga_latent_mix_fwd: null argument");
  GA_CHECK(q->c >= zdim && z->c >= zdim, "ga_latent_mix_fwd: channel counts smaller than zdim");
  GA_CHECK(q->n == z->n && q->h == z->h && q->w == z->w, "ga_latent_mix_fwd: shape mismatch");
  GA_CHECK(!p || (p->c == 2 * zdim && p->n == q->n && p->h == q->h && p->w == q->w), "ga_latent_mix_fwd: prior tensor must have 2*zdim channels");
  const int64_t total_pix = (int64_t)z->n * z->h * z->w;
  if (total_pix == 0) return 0;
  if ((zdim & 3) == 0 && (q->c & 3) == 0 && (z->c & 3) == 0) {
    latent_mix_vec4_kernel<<<cdiv(total_pix * (z->c / 4), 256), 256, 0, (cudaStream_t)stream>>>(
        q->data, q->dtype, q->c, p ? p->data : nullptr, p ? p->dtype : GA_F32, eps, make_seed(seed, (cudaStream_t)stream), level, sample0, alpha_dev,
        temperature, zdim, total_pix, z->h * z->w, z->data, z->dtype, z->c);
    GA_LAUNCH_OK();
    return 0;
  }
  latent_mix_kernel<<<cdiv(total_pix, 128), 128, 0, (cudaStream_t)stream>>>(
      q->data, q->dtype, q->c, p ? p->data : nullptr, p ? p->dtype : GA_F32, eps, make_seed(seed, (cudaStream_t)stream), level, sample0, alpha_dev,
      temperature, zdim, total_pix, z->h * z->w, z->data, z->dtype, z->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_discmix_mean_fwd(const ga_tensor* logits, int n_mix, float* purified, const ga_tensor* cls, void* stream) {
  GA_CHECK(logits && purified && n_mix > 0, "ga_discmix_mean_fwd: null argument");
  GA_CHECK(logits->c == 10 * n_mix, "ga_discmix_mean_fwd: logits must have 10*n_mix channels (3-channel images)");
  GA_CHECK(!cls || (cls->c == 3 && cls->n == logits->n && cls->h == logits->h && cls->w == logits->w), "ga_discmix_mean_fwd: classifier input must be NHWC with 3 channels");
  const int64_t total_pix = (int64_t)logits->n * logits->h * logits->w;
  if (total_pix == 0) return 0;
  const size_t smem = (size_t)DM_PIX * (10 * n_mix + 1) * sizeof(float);
  GA_CHECK(smem <= 200 * 1024, "ga_discmix_mean_fwd: too many mixtures");
  static size_t configured = 0;
  if (configured < smem) {
    GA_CUDA(cudaFuncSetAttribute(discmix_mean_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  discmix_mean_kernel<<<cdiv(total_pix, DM_PIX), 128, smem, (cudaStream_t)stream>>>(
      logits->data, logits->dtype, n_mix, logits->h * logits->w, total_pix, purified, cls ? cls->data : nullptr,
      cls ? cls->dtype : GA_F32);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_upsample_nearest2x(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && out->h == 2 * in->h && out->w == 2 * in->w && out->c == in->c && out->n == in->n && (in->c % 4) == 0,
           "ga_upsample_nearest2x: shape mismatch");
  const int64_t total = numel(out) / 4;
  if (total == 0) return 0;
  upsample_nearest2x_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, out->data, out->dtype, in->n, in->h, in->w, in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_upsample_bilinear2x(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && out->h == 2 * in->h && out->w == 2 * in->w && out->c == in->c && out->n == in->n && (in->c % 4) == 0,
           "ga_upsample_bilinear2x: shape mismatch");
  const int64_t total = numel(out) / 4;
  if (total == 0) return 0;
  upsample_bilinear2x_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, out->data, out->dtype, in->n, in->h, in->w, in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_maxpool2x2(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && out->h == in->h / 2 && out->w == in->w / 2 && out->c == in->c && out->n == in->n && (in->c % 4) == 0,
           "ga_maxpool2x2: shape mismatch");
  const int64_t total = numel(out) / 4;
  if (total == 0) return 0;
  maxpool2x2_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, out->data, out->dtype, in->n, in->h, in->w, in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_subsample2x(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && out->h == (in->h + 1) / 2 && out->w == (in->w + 1) / 2 && out->c == in->c && out->n == in->n && (in->c % 4) == 0,
           "ga_subsample2x: shape mismatch");
  const int64_t total = numel(out) / 4;
  if (total == 0) return 0;
  subsample2x_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, out->data, out->dtype, in->n, in->h, in->w, in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_maxpool3x3s2(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && out->h == (in->h - 1) / 2 + 1 && out->w == (in->w - 1) / 2 + 1 && out->c == in->c && out->n == in->n && (in->c % 4) == 0,
           "ga_maxpool3x3s2: shape mismatch");
  const int64_t total = numel(out) / 4;
  if (total == 0) return 0;
  maxpool3x3s2_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, out->data, out->dtype, in->n, in->h, in->w, in->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_global_avgpool(const ga_tensor* in, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && out->n == in->n && out->h == 1 && out->w == 1 && out->c == in->c, "ga_global_avgpool: shape mismatch");
  if (numel(in) == 0) return 0;
  global_avgpool_kernel<<<in->n, 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, in->h * in->w, in->c, out->data, out->dtype);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_affine_act(const ga_tensor* in, const float* scale, const float* shift, int act, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && same_shape(in, out), "ga_affine_act: shape mismatch");
  GA_CHECK((scale == nullptr) == (shift == nullptr), "ga_affine_act: scale and shift go together");
  const int64_t total = numel(in);
  if (total == 0) return 0;
  const int rtf = (out->dtype == GA_F32 && round_tf32_enabled()) ? 1 : 0;
  if ((in->c & 7) == 0)
    affine_act_vec8_kernel<<<cdiv(total / 8, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, scale, shift, act, out->data, out->dtype, in->c, total / 8, rtf);
  else
    affine_act_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, scale, shift, act, out->data, out->dtype, in->c, total, rtf);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_cast(const ga_tensor* in, const ga_tensor* out, void* stream) {
  return ga_affine_act(in, nullptr, nullptr, GA_ACT_NONE, out, stream);
}

extern "C" int ga_nchw_to_nhwc(const float* in, const ga_tensor* out, float scale, float shift, void* stream) {
  GA_CHECK(in && out, "ga_nchw_to_nhwc: null argument");
  const int64_t total = numel(out);
  if (total == 0) return 0;
  nchw_to_nhwc_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in, out->data, out->dtype, scale, shift, out->n, out->c, out->h, out->w);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_pgd_linf_step(float* x_adv, const float* grad, const float* x_nat, float step, float eps, int64_t numel_, void* stream) {
  GA_CHECK(x_adv && grad && x_nat && numel_ >= 0, "ga_pgd_linf_step: null argument");
  if (numel_ == 0) return 0;
  GA_CHECK(((((uintptr_t)x_adv) | ((uintptr_t)grad) | ((uintptr_t)x_nat)) & 15) == 0, "ga_pgd_linf_step: buffers must be 16-byte aligned");
  const int64_t n4 = numel_ / 4;
  pgd_linf_step_kernel<<<max(1, cdiv(n4, 256)), 256, 0, (cudaStream_t)stream>>>(x_adv, grad, x_nat, step, eps, n4, numel_);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_softmax_xent(const float* logits, const int64_t* labels, int n, int classes, float* loss, float* dlogits,
                               int32_t* pred, unsigned long long* n_correct, void* stream) {
  GA_CHECK(logits && n >= 0 && classes > 0, "ga_softmax_xent: bad arguments");
  if (n == 0) return 0;
  softmax_xent_kernel<<<cdiv((int64_t)n * 32, 256), 256, 0, (cudaStream_t)stream>>>(logits, labels, n, classes, loss, dlogits, pred, n_correct);
  GA_LAUNCH_OK();
  return 0;
}
