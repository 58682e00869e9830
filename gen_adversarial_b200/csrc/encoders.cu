// Encoder-side pieces of the StyleGAN purifiers (SURVEY rows A13, A17, A18) that are not convolutions:
//   * LayerNorm(x + y), multi-head attention with 16 learned queries  -- DETR-style TransformerDecoderLayer of the
//     Style-Transformer encoder (StyleGan_Trans/models/transformer.py:17-100, nn.MultiheadAttention d=512, 4 heads)
//   * W+ code assembly: w0 repeated + per-level deltas + latent_avg   (StyleGan_E4E/encoding/encoder.py:125-139, psp.py:92-99)
//   * bilinear resize with a row crop (kornia.geometry.resize, align_corners=False; models.py:307-308)
//   * image output: k x k face_pool, row masking with -1, second 2x2 mean (= bilinear /2), denormalise, NCHW + NHWC
//     (psp.py:26,114; models.py:346-351; abstract_models.py:184-185)
//   * Philox N(0,1) fill for the style noise of the latent interpolation (models.py:119,334)
// All are HBM- or latency-bound; linear layers around them run on the conv kernels as 1x1 convolutions.
#include "ga_common.cuh"

namespace ga {

__device__ __forceinline__ float ld1e(const void* base, int dtype, int64_t off) {
  return dtype == GA_F32 ? reinterpret_cast<const float*>(base)[off]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[off]);
}
__device__ __forceinline__ void st1e(void* base, int dtype, int64_t off, float v) {
  if (dtype == GA_F32) reinterpret_cast<float*>(base)[off] = v;
  else reinterpret_cast<__nv_bfloat16*>(base)[off] = __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------------------- out = LayerNorm(x + y) * gamma + beta : one warp per row
__global__ void __launch_bounds__(256) add_layernorm_kernel(const void* x, int x_dtype, const void* y, int y_dtype,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                                            int rows, int d, void* out, int out_dtype, void* out2, int out2_dtype) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int64_t base = (int64_t)row * d;
  float s = 0.f;
  for (int i = lane; i < d; i += 32) s += ld1e(x, x_dtype, base + i) + (y != nullptr ? ld1e(y, y_dtype, base + i) : 0.f);
  const float mean = warp_sum(s) / (float)d;
  float v = 0.f;
  for (int i = lane; i < d; i += 32) {
    const float t = ld1e(x, x_dtype, base + i) + (y != nullptr ? ld1e(y, y_dtype, base + i) : 0.f) - mean;
    v = fmaf(t, t, v);
  }
  const float rstd = rsqrtf(warp_sum(v) / (float)d + eps);      // biased variance (torch.nn.LayerNorm)
  for (int i = lane; i < d; i += 32) {
    const float t = ld1e(x, x_dtype, base + i) + (y != nullptr ? ld1e(y, y_dtype, base + i) : 0.f);
    const float o = (t - mean) * rstd * gamma[i] + beta[i];
    st1e(out, out_dtype, base + i, o);
    if (out2 != nullptr) st1e(out2, out2_dtype, base + i, o);
  }
}

// ---------------------------------------------------------------------------- attention, pass 1: scaled scores
// q: [B][Q][q_stride] (head h at column q_off + h*dh), k: [B][S][k_stride] (k_off + h*dh)  ->  scores[B][H][Q][S] fp32
// one CTA per (key tile of 64, head, batch); the Q rows of the head sit in shared memory
template <int DH>
__global__ void __launch_bounds__(256) attn_scores_kernel(const void* q, int q_dtype, int q_stride, int q_off, const void* k, int k_dtype,
                                                          int k_stride, int k_off, int Q, int S, int H, float scale, float* __restrict__ scores) {
  extern __shared__ float sm[];
  float* s_q = sm;                 // [Q][DH]
  float* s_k = sm + Q * DH;        // [64][DH + 1]
  const int b = blockIdx.z, h = blockIdx.y, s0 = blockIdx.x * 64;
  for (int i = threadIdx.x; i < Q * DH; i += 256) {
    const int qi = i / DH, d = i - qi * DH;
    s_q[i] = ld1e(q, q_dtype, ((int64_t)b * Q + qi) * q_stride + q_off + h * DH + d) * scale;
  }
  for (int i = threadIdx.x; i < 64 * DH; i += 256) {
    const int si = i / DH, d = i - si * DH;
    s_k[si * (DH + 1) + d] = (s0 + si < S) ? ld1e(k, k_dtype, ((int64_t)b * S + s0 + si) * k_stride + k_off + h * DH + d) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < Q * 64; i += 256) {
    const int qi = i >> 6, si = i & 63;
    if (s0 + si >= S) continue;
    float a = 0.f;
#pragma unroll 8
    for (int d = 0; d < DH; ++d) a = fmaf(s_q[qi * DH + d], s_k[si * (DH + 1) + d], a);
    scores[(((int64_t)b * H + h) * Q + qi) * S + s0 + si] = a;
  }
}

// ---------------------------------------------------------------------------- attention, pass 2: softmax over S, then P.V
// one CTA per (head, batch): row max / sum by one warp per query row (fixed order), P.V with a thread per (query, 8 dims)
template <int DH>
__global__ void __launch_bounds__(256) attn_pv_kernel(float* __restrict__ scores, const void* v, int v_dtype, int v_stride, int v_off, int Q,
                                                      int S, int H, void* out, int out_dtype, int out_stride) {
  extern __shared__ float sm[];
  float* s_v = sm;                   // [64][DH]
  float* s_p = sm + 64 * DH;         // [Q][64]
  float* s_inv = s_p + Q * 64;       // [Q]
  const int b = blockIdx.y, h = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sc = scores + ((int64_t)b * H + h) * Q * S;
  for (int qi = warp; qi < Q; qi += 8) {
    float m = -INFINITY;
    for (int s = lane; s < S; s += 32) m = fmaxf(m, sc[(int64_t)qi * S + s]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int s = lane; s < S; s += 32) {
      const float e = expf(sc[(int64_t)qi * S + s] - m);
      sc[(int64_t)qi * S + s] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    if (lane == 0) s_inv[qi] = 1.f / sum;
  }
  __syncthreads();
  // thread -> (query, dim group): Q * DH / 8 items, 8 consecutive dims each
  constexpr int GROUPS = DH / 8;
  const int items = Q * GROUPS;
  float acc[2][8];
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[u][j] = 0.f;
  for (int s0 = 0; s0 < S; s0 += 64) {
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * DH; i += 256) {
      const int si = i / DH, d = i - si * DH;
      s_v[i] = (s0 + si < S) ? ld1e(v, v_dtype, ((int64_t)b * S + s0 + si) * v_stride + v_off + h * DH + d) : 0.f;
    }
    for (int i = threadIdx.x; i < Q * 64; i += 256) {
      const int qi = i >> 6, si = i & 63;
      s_p[i] = (s0 + si < S) ? sc[(int64_t)qi * S + s0 + si] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int it = threadIdx.x + u * 256;
      if (it >= items) continue;
      const int qi = it / GROUPS, d0 = (it - qi * GROUPS) * 8;
      for (int si = 0; si < 64; ++si) {
        const float pv = s_p[qi * 64 + si];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[u][j] = fmaf(pv, s_v[si * DH + d0 + j], acc[u][j]);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int it = threadIdx.x + u * 256;
    if (it >= items) continue;
    const int qi = it / GROUPS, d0 = (it - qi * GROUPS) * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) st1e(out, out_dtype, ((int64_t)b * Q + qi) * out_stride + h * DH + d0 + j, acc[u][j] * s_inv[qi]);
  }
}

// ---------------------------------------------------------------------------- W+ code assembly
// heads: [L][B][D] (head-major, what the map2style heads write);  out[b][l][:] = heads[0][b] (if use_w0 and l > 0) + heads[l][b] + avg[l]
// with use_w0 = 0 and heads laid out [B][L][D] (heads_lb = 0) this is `codes + latent_avg` of the Style-Transformer.
__global__ void codes_assemble_kernel(const float* __restrict__ heads, int heads_lb, int use_w0, const float* __restrict__ avg, int B, int L,
                                      int D, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * L * D) return;
  const int d = (int)(i % D);
  const int l = (int)((i / D) % L);
  const int64_t b = i / ((int64_t)D * L);
  float v = heads_lb ? heads[((int64_t)l * B + b) * D + d] : heads[i];
  if (use_w0 && l > 0) v += heads_lb ? heads[b * D + d] : heads[(b * L) * D + d];
  if (avg != nullptr) v += avg[(int64_t)l * D + d];
  out[i] = v;
}

// adjoint of codes_assemble (heads_lb, use_w0): g_heads[l][b][d] = g_codes[b][l][d] (l > 0), g_heads[0][b][d] = sum_l g_codes[b][l][d]
// in increasing l (one thread per (b, d): fixed order, no atomics, independent of the batch size)
__global__ void codes_assemble_bwd_kernel(const float* __restrict__ g, int B, int L, int D, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * D) return;
  const int d = (int)(i % D);
  const int64_t b = i / D;
  const float* gb = g + b * L * D + d;
  float s = 0.f;
  for (int l = 0; l < L; ++l) {
    const float v = gb[(int64_t)l * D];
    s += v;
    if (l > 0) out[((int64_t)l * B + b) * D + d] = v;
  }
  out[b * D + d] = s;
}

// ---------------------------------------------------------------------------- bilinear resize (align_corners=False, no antialias) + row crop
// out[n, y, x, c] = bilinear(in[n], (y + crop_y0 + 0.5) * H/Hfull - 0.5, (x + 0.5) * W/Wo - 0.5)   (F.interpolate semantics)
__global__ void resize_bilinear_kernel(const void* in, int in_dtype, int N, int H, int W, int C, int Hfull, int crop_y0, int Ho, int Wo,
                                       void* out, int out_dtype) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * Ho * Wo * C) return;
  const int c = (int)(idx % C);
  int64_t t = idx / C;
  const int x = (int)(t % Wo); t /= Wo;
  const int y = (int)(t % Ho);
  const int64_t n = t / Ho;
  const float sy = (float)H / (float)Hfull, sx = (float)W / (float)Wo;
  const float fy = fmaxf(((float)(y + crop_y0) + 0.5f) * sy - 0.5f, 0.f);
  const float fx = fmaxf(((float)x + 0.5f) * sx - 0.5f, 0.f);
  const int y0 = min((int)fy, H - 1), x0 = min((int)fx, W - 1);
  const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
  const float ly = fy - (float)y0, lx = fx - (float)x0;
  const float v00 = ld1e(in, in_dtype, ((n * H + y0) * W + x0) * C + c), v01 = ld1e(in, in_dtype, ((n * H + y0) * W + x1) * C + c);
  const float v10 = ld1e(in, in_dtype, ((n * H + y1) * W + x0) * C + c), v11 = ld1e(in, in_dtype, ((n * H + y1) * W + x1) * C + c);
  const float o = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
  st1e(out, out_dtype, idx, o);
}

// ---------------------------------------------------------------------------- generator image -> boundary tensors
// in: NHWC (N, S, S, C>=3) fp32 image in [-1, 1] (4th channel = padding).  stage 1: k1 x k1 mean (face_pool); stage 2 (k2 = 2 only):
// rows r < mask_rows or r >= S/k1 - mask_rows of the pooled image are set to -1, then a 2x2 mean (= bilinear resize by 1/2).
// purified_nchw (N,3,So,So) = o * out_scale + out_shift (kornia denormalize);  cls_nhwc (N,So,So,3) = o (the classifier normalises with
// the same mean/std, so it consumes the un-denormalised value).
__global__ void image_pool_out_kernel(const float* __restrict__ in, int N, int S, int C, int k1, int k2, int mask_rows, float out_scale,
                                      float out_shift, float* __restrict__ purified, void* cls, int cls_dtype) {
  const int Sp = S / k1, So = Sp / k2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;        // over (n, y, x)
  if (idx >= (int64_t)N * So * So) return;
  const int x = (int)(idx % So);
  const int y = (int)((idx / So) % So);
  const int64_t n = idx / ((int64_t)So * So);
  float acc[3] = {0.f, 0.f, 0.f};
  for (int py = 0; py < k2; ++py) {
    const int r = y * k2 + py;
    const bool masked = r < mask_rows || r >= Sp - mask_rows;
    for (int px = 0; px < k2; ++px) {
      const int q = x * k2 + px;
      float a[3] = {0.f, 0.f, 0.f};
      if (masked) { a[0] = a[1] = a[2] = -1.f; }
      else {
        for (int dy = 0; dy < k1; ++dy)
          for (int dx = 0; dx < k1; ++dx) {
            const float* p = in + ((n * S + r * k1 + dy) * S + q * k1 + dx) * C;
            a[0] += p[0]; a[1] += p[1]; a[2] += p[2];
          }
        const float inv = 1.f / (float)(k1 * k1);
        a[0] *= inv; a[1] *= inv; a[2] *= inv;
      }
      acc[0] += a[0]; acc[1] += a[1]; acc[2] += a[2];
    }
  }
  const float inv2 = 1.f / (float)(k2 * k2);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float o = acc[c] * inv2;
    if (purified != nullptr) purified[((n * 3 + c) * So + y) * So + x] = fmaf(o, out_scale, out_shift);
    if (cls != nullptr) st1e(cls, cls_dtype, idx * 3 + c, o);
  }
}

// ---------------------------------------------------------------------------- N(0, std) fill, keyed by (seed, code index, global sample index)
// out[l][b][d] (the reference's torch.normal(0, std, (n_codes, b, d)) layout)
__global__ void philox_codes_kernel(SeedArg seed_arg, int64_t sample0, float std_, int L, int B, int D, float* __restrict__ out) {
  const uint64_t seed = seed_arg.get();
  const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;          // D % 4 == 0
  const int d4n = D >> 2;
  if (i4 >= (int64_t)L * B * d4n) return;
  const int d4 = (int)(i4 % d4n);
  const int b = (int)((i4 / d4n) % B);
  const int l = (int)(i4 / ((int64_t)d4n * B));
  float z[4];
  philox_normal4(seed, 0x5747u + (uint64_t)l, (uint64_t)(sample0 + b) * d4n + d4, z);
  *reinterpret_cast<float4*>(out + i4 * 4) = make_float4(z[0] * std_, z[1] * std_, z[2] * std_, z[3] * std_);
}

}  // namespace ga

using namespace ga;

extern "C" int ga_add_layernorm(const ga_tensor* x, const ga_tensor* y, const float* gamma, const float* beta, float eps,
                                const ga_tensor* out, const ga_tensor* out2, void* stream) {
  GA_CHECK(x && gamma && beta && out && same_shape(x, out), "ga_add_layernorm: bad arguments");
  GA_CHECK(!y || same_shape(x, y), "ga_add_layernorm: y shape mismatch");
  GA_CHECK(!out2 || same_shape(x, out2), "ga_add_layernorm: out2 shape mismatch");
  const int64_t rows = (int64_t)x->n * x->h * x->w;
  if (rows == 0) return 0;
  add_layernorm_kernel<<<cdiv(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(x->data, x->dtype, y ? y->data : nullptr, y ? y->dtype : GA_F32,
                                                                                gamma, beta, eps, (int)rows, x->c, out->data, out->dtype,
                                                                                out2 ? out2->data : nullptr, out2 ? out2->dtype : GA_F32);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int64_t ga_attention_ws_floats(int b, int heads, int q, int s) { return (int64_t)b * heads * q * s; }

extern "C" int ga_attention(const ga_tensor* q, int q_off, const ga_tensor* k, int k_off, const ga_tensor* v, int v_off, int heads, int dh,
                            float* scores_ws, const ga_tensor* out, void* stream) {
  GA_CHECK(q && k && v && out && scores_ws, "ga_attention: null argument");
  GA_CHECK(dh == 128, "ga_attention: head dim %d not supported (128 only)", dh);
  const int B = q->n, Q = q->h * q->w, S = k->h * k->w;
  GA_CHECK(k->n == B && v->n == B && v->h * v->w == S && out->n == B && out->h * out->w == Q && out->c == heads * dh,
           "ga_attention: shape mismatch");
  GA_CHECK(q_off + heads * dh <= q->c && k_off + heads * dh <= k->c && v_off + heads * dh <= v->c, "ga_attention: column window out of range");
  GA_CHECK(Q >= 1 && Q <= 32, "ga_attention: %d queries (1..32 supported)", Q);
  if (B == 0 || S == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const float scale = 1.0f / sqrtf((float)dh);
  const size_t smem1 = ((size_t)Q * 128 + 64 * 129) * sizeof(float);
  const size_t smem2 = ((size_t)64 * 128 + Q * 64 + Q) * sizeof(float);
  static bool configured = false;
  if (!configured) {
    GA_CUDA(cudaFuncSetAttribute(attn_scores_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (32 * 128 + 64 * 129) * 4));
    GA_CUDA(cudaFuncSetAttribute(attn_pv_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (64 * 128 + 32 * 64 + 32) * 4));
    configured = true;
  }
  attn_scores_kernel<128><<<dim3(cdiv(S, 64), heads, B), 256, smem1, s>>>(q->data, q->dtype, q->c, q_off, k->data, k->dtype, k->c, k_off, Q, S,
                                                                         heads, scale, scores_ws);
  GA_LAUNCH_OK();
  attn_pv_kernel<128><<<dim3(heads, B), 256, smem2, s>>>(scores_ws, v->data, v->dtype, v->c, v_off, Q, S, heads, out->data, out->dtype, out->c);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_codes_assemble(const float* heads, int heads_lb, int use_w0, const float* latent_avg, int b, int l, int d, float* out,
                                 void* stream) {
  GA_CHECK(heads && out && b >= 0 && l > 0 && d > 0, "ga_codes_assemble: bad arguments");
  const int64_t total = (int64_t)b * l * d;
  if (total == 0) return 0;
  codes_assemble_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(heads, heads_lb, use_w0, latent_avg, b, l, d, out);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_codes_assemble_bwd(const float* g_codes, int b, int l, int d, float* g_heads, void* stream) {
  GA_CHECK(g_codes && g_heads && b >= 0 && l >= 1 && d >= 1, "ga_codes_assemble_bwd: bad arguments");
  const int64_t total = (int64_t)b * d;
  if (total == 0) return 0;
  codes_assemble_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(g_codes, b, l, d, g_heads);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_resize_bilinear(const ga_tensor* in, int full_h, int crop_y0, const ga_tensor* out, void* stream) {
  GA_CHECK(in && out && in->n == out->n && in->c == out->c && full_h >= 1 && crop_y0 >= 0 && crop_y0 + out->h <= full_h,
           "ga_resize_bilinear: bad arguments");
  const int64_t total = numel(out);
  if (total == 0) return 0;
  resize_bilinear_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(in->data, in->dtype, in->n, in->h, in->w, in->c, full_h, crop_y0,
                                                                             out->h, out->w, out->data, out->dtype);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_image_pool_out(const ga_tensor* in, int k1, int k2, int mask_rows, float out_scale, float out_shift, float* purified_nchw,
                                 const ga_tensor* cls_nhwc, void* stream) {
  GA_CHECK(in && in->dtype == GA_F32 && in->h == in->w && in->c >= 3 && k1 >= 1 && (k2 == 1 || k2 == 2) && in->h % (k1 * k2) == 0 &&
               mask_rows >= 0 && (purified_nchw || cls_nhwc),
           "ga_image_pool_out: bad arguments");
  const int so = in->h / (k1 * k2);
  GA_CHECK(!cls_nhwc || (cls_nhwc->n == in->n && cls_nhwc->h == so && cls_nhwc->w == so && cls_nhwc->c == 3), "ga_image_pool_out: cls shape mismatch");
  const int64_t total = (int64_t)in->n * so * so;
  if (total == 0) return 0;
  image_pool_out_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>((const float*)in->data, in->n, in->h, in->c, k1, k2, mask_rows,
                                                                            out_scale, out_shift, purified_nchw,
                                                                            cls_nhwc ? cls_nhwc->data : nullptr, cls_nhwc ? cls_nhwc->dtype : GA_F32);
  GA_LAUNCH_OK();
  return 0;
}

extern "C" int ga_philox_codes(uint64_t seed, int64_t sample0, float std_, int l, int b, int d, float* out, void* stream) {
  GA_CHECK(out && l > 0 && b >= 0 && d > 0 && d % 4 == 0, "ga_philox_codes: bad arguments");
  const int64_t total4 = (int64_t)l * b * (d / 4);
  if (total4 == 0) return 0;
  philox_codes_kernel<<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(make_seed(seed, (cudaStream_t)stream), sample0, std_, l, b, d, out);
  GA_LAUNCH_OK();
  return 0;
}
