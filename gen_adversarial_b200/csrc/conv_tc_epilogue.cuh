// Epilogue of the tcgen05 convolution kernels (conv_tc.cu, conv3x3_tc.cu): one 128-row x BLOCK_N accumulator tile
//   TMEM -> registers -> + bias -> activation (+ saved derivative) -> + add -> * f(mul) -> bf16 / fp32 (TF32-rounded on request)
//   -> swizzled staging tile in shared memory -> TMA store   (or direct vector stores for odd shapes / partial tiles).
// Called by the 4 epilogue warps of a CTA (warp quadrant q = warp & 3 owns TMEM lanes 32q..32q+31 = tile rows).
#pragma once
#include "ga_common.cuh"
#include "tc_ptx.cuh"

namespace ga {

struct TcParams {
  int taps, kw, pad, stride;  // filter taps of source 1; stride 1 or 2 (TMA element strides do the decimation)
  int k32;                    // 1: 32-channel K blocks (64-byte swizzle) for Cin = 32, 96, ...: no half-empty 64-channel boxes
  int tf32;                   // 1: fp32 activations and weights, kind::tf32 MMA, 32-channel K blocks (32 x 4 B = one 128-byte swizzle row)
  int cin, kc1, kc2;          // channels of source 1, its 64-blocks per tap, 64-blocks of source 2
  int bw, bh, bn;             // pixel box of one M tile (bw*bh*bn == 128)
  int tiles_x, tiles_y;       // tiles per image row / column (bn == 1) -- else whole images per tile
  int H, W;
  int64_t M;                  // total output pixels
  int cout;
  int n_blocks;               // output-channel blocks (grid = m_tiles * n_blocks, N block fastest)
  const float* bias;
  int post_act;
  const void* add; int add_dtype;
  __nv_bfloat16* out_bf16;
  float* out_f32;
  int tma_store;              // 1: epilogue stages the tile in (swizzled) shared memory and TMA-stores it
  int partial;                // 1: the last tile row of an image hangs over its bottom edge (bn == 1, bw == W): mask rows, direct stores
  const void* mul; int mul_dtype, mul_mode;   // backward: out = (act(acc+bias) + add) * f(mul)
  __nv_bfloat16* dact;        // taping forward: derivative of post_act at the pre-activation (bf16)
  const float* act_slope;     // PReLU slopes [cout]
  int act_after_add;          // act(acc + bias + add)
  int round_tf32;             // fp32 output rounded to TF32 (feeds a kind::tf32 conv)
  float* csum;                // optional (persistent 3x3 kernel, lean epilogue): per-image channel sums of the bf16 output in 128-pixel
                              // slices, [n][HW / 128][cout] -- the layout ga_channel_sum writes (SE squeeze fused into the conv)
};

// conv3x3_tc.cu: persistent halo-reuse kernel for 3x3 / stride 1 / pad 1; -> 0 launched, 1 error, -1 shape not covered
int conv3x3_halo_launch(const ga_tensor* in, const void* weight, int ktot, const ga_tensor* out_bf16, const ga_tensor* out_f32, TcParams p,
                        cudaStream_t s);
int conv1x1_persistent_launch(const ga_tensor* in, const void* weight, int ktot, const ga_tensor* out_bf16, const ga_tensor* out_f32, TcParams p,
                              cudaStream_t s);
bool conv3x3_halo_csum_ok(const ga_tensor* in, int cout, const TcParams& p, bool out_b, bool out_f);

// tmem_acc: TMEM address (lane 0) of column 0 of the accumulator; pix0: global index of the tile's first output pixel; row_limit: rows of
// the tile that exist (128, or fewer for the partial last tile row of an image); stage: 1024-aligned staging memory (TMA-store mode);
// s_bias / s_slope: BLOCK_N floats each in shared memory (bias and PReLU slopes of this N block; GENERAL_ACT only).  The slopes serve
// post_act = GA_ACT_PRELU and mul_mode = GA_MUL_PRELU_FROM_Y alike: the host runs both on GENERAL_ACT instantiations.
// DEFER_STORE_WAIT: return without waiting for the bulk stores to have read the staging tile (the caller waits before re-using it).
// LD_COLS: accumulator columns fetched per tcgen05.ld round trip.  A round trip costs ~1k cycles while the tensor pipe is busy (measured: the
// persistent 3x3 kernel spent 1000 clk per 16-column chunk); a kernel with few resident warps must put many columns in flight per wait.
template <int BLOCK_N, bool GENERAL_ACT, bool DEFER_STORE_WAIT = false, int LD_COLS = 16>
__device__ __forceinline__ void tc_epilogue_tile(const TcParams& p, const CUtensorMap* tmOutB, const CUtensorMap* tmOutF,
                                                 const CUtensorMap* tmOutD, uint32_t tmem_acc, int n_blk, int64_t pix0, int row_limit,
                                                 uint8_t* stage, const float* s_bias, const float* s_slope, int q, int lane) {
  const int row = q * 32 + lane;
  const int64_t pix = pix0 + row;
  // partial tiles (H not a multiple of the tile's row count): rows past the image's last row were zero-filled by TMA, never stored
  const bool row_ok = pix < p.M && row < row_limit;
  const bool vec_ok = (p.cout & 7) == 0;
  // staging tiles for the TMA store re-use the (now idle) operand ring: every MMA has retired, so every TMA load
  // has landed and every operand read is done.  Layout = the SWIZZLE_128B box layout of the output tensor maps:
  // 128-byte row panels (64 bf16 / 32 fp32 columns), 16-byte chunk index XOR (row & 7).
  uint8_t* stage_b = stage;                                  // bf16: BLOCK_N/64 panels x 128 rows x 128 B
  uint8_t* stage_f = stage + (p.out_bf16 != nullptr ? ((BLOCK_N + 63) / 64) * 16384 : 0);   // fp32: BLOCK_N/32 panels of 16 KB
  uint8_t* stage_d = stage_f + (p.out_f32 != nullptr ? (BLOCK_N / 32) * 16384 : 0);               // bf16 dact panels
  const uint32_t sw = (uint32_t)(row & 7);
#pragma unroll 1
  for (int cg = 0; cg < BLOCK_N; cg += LD_COLS) {
  uint32_t rr[LD_COLS / 16][16];
#pragma unroll
  for (int i = 0; i < LD_COLS / 16; ++i)
    if (cg + i * 16 < BLOCK_N) tmem_ld16(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg + i * 16), rr[i]);
  tmem_ld_wait();
#pragma unroll
  for (int ci = 0; ci < LD_COLS / 16; ++ci) {
    const int c0 = cg + ci * 16;
    if (c0 >= BLOCK_N) break;
    uint32_t (&r)[16] = rr[ci];
    const int nb = n_blk * BLOCK_N + c0;
    if (nb >= p.cout) continue;                              // whole chunk beyond Cout (warp-uniform)
    float v[16];
    const int64_t off = pix * p.cout + nb;
    const bool full = vec_ok && nb + 16 <= p.cout;
    bool have_v = false;
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]) + s_bias[c0 + j];
    if (p.dact != nullptr && (row_ok || p.tma_store)) {   // save act'(pre-activation) for the backward pass
      float dv[16];
      if (!GENERAL_ACT && p.post_act == GA_ACT_SILU) { silu_with_grad_fast_n<16>(v, v, dv); have_v = true; }   // one tanh for both, in place
      else act_grad_fast_n<16>(v, dv, p.post_act);         // dact is bf16
      if (p.tma_store) {
        uint8_t* panel = stage_d + (c0 >> 6) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 63) >> 3);
        *reinterpret_cast<uint4*>(panel + (((k0) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(dv[0], dv[1]), pack_bf16x2(dv[2], dv[3]), pack_bf16x2(dv[4], dv[5]), pack_bf16x2(dv[6], dv[7]));
        *reinterpret_cast<uint4*>(panel + (((k0 + 1) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(dv[8], dv[9]), pack_bf16x2(dv[10], dv[11]), pack_bf16x2(dv[12], dv[13]), pack_bf16x2(dv[14], dv[15]));
      } else if (full) {
        uint4* o = reinterpret_cast<uint4*>(p.dact + off);
        o[0] = make_uint4(pack_bf16x2(dv[0], dv[1]), pack_bf16x2(dv[2], dv[3]), pack_bf16x2(dv[4], dv[5]), pack_bf16x2(dv[6], dv[7]));
        o[1] = make_uint4(pack_bf16x2(dv[8], dv[9]), pack_bf16x2(dv[10], dv[11]), pack_bf16x2(dv[12], dv[13]), pack_bf16x2(dv[14], dv[15]));
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (nb + j < p.cout) p.dact[off + j] = __float2bfloat16_rn(dv[j]);
      }
    }
    if (have_v) {
    } else if (!GENERAL_ACT) {
      apply_act_fast_n<16>(v, p.post_act);
    } else if (!p.act_after_add) {
      if (p.post_act == GA_ACT_PRELU) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = v[j] > 0.f ? v[j] : s_slope[c0 + j] * v[j];
      } else {
        apply_act_fast_n<16>(v, p.post_act);
      }
    }
    if (p.add != nullptr && row_ok) {
      if (full) {
        if (p.add_dtype == GA_F32) {
          const float4* a4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.add) + off);
#pragma unroll
          for (int j = 0; j < 4; ++j) { float4 t = __ldg(a4 + j); v[4 * j] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w; }
        } else {
          const uint4* a4 = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.add) + off);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint4 t = __ldg(a4 + j);
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[k]);
              v[8 * j + 2 * k] += __low2float(h); v[8 * j + 2 * k + 1] += __high2float(h);
            }
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (nb + j < p.cout)
            v[j] += (p.add_dtype == GA_F32) ? reinterpret_cast<const float*>(p.add)[off + j]
                                            : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.add)[off + j]);
      }
    }
    if (GENERAL_ACT && p.act_after_add) {
      if (p.post_act == GA_ACT_PRELU) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = v[j] > 0.f ? v[j] : s_slope[c0 + j] * v[j];
      } else {
        apply_act_fast_n<16>(v, p.post_act);
      }
    }
    if (p.mul != nullptr && row_ok && full) {
      float mv[16];
      if (p.mul_dtype == GA_F32) {
        const float4* m4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.mul) + off);
#pragma unroll
        for (int j = 0; j < 4; ++j) { float4 t = __ldg(m4 + j); mv[4 * j] = t.x; mv[4 * j + 1] = t.y; mv[4 * j + 2] = t.z; mv[4 * j + 3] = t.w; }
      } else {
        const uint4* m4 = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.mul) + off);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          uint4 t = __ldg(m4 + j);
          const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[k]);
            mv[8 * j + 2 * k] = __low2float(h); mv[8 * j + 2 * k + 1] = __high2float(h);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] *= mul_factor(mv[j], p.mul_mode, GENERAL_ACT ? s_slope[c0 + j] : 0.f);
    } else if (p.mul != nullptr && row_ok) {
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        if (nb + j < p.cout) {
          const float mv = (p.mul_dtype == GA_F32) ? __ldg(reinterpret_cast<const float*>(p.mul) + off + j)
                                                   : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.mul)[off + j]);
          v[j] *= mul_factor(mv, p.mul_mode, GENERAL_ACT ? s_slope[c0 + j] : 0.f);
        }
      }
    }
    float vf[16];                                            // fp32 output values (TF32-rounded on request)
#pragma unroll
    for (int j = 0; j < 16; ++j) vf[j] = (p.round_tf32 && p.out_f32 != nullptr) ? round_tf32(v[j]) : v[j];
    if (p.tma_store) {
      if (p.out_bf16 != nullptr) {
        uint8_t* panel = stage_b + (c0 >> 6) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 63) >> 3);
        *reinterpret_cast<uint4*>(panel + (((k0) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        *reinterpret_cast<uint4*>(panel + (((k0 + 1) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
      }
      if (p.out_f32 != nullptr) {
        uint8_t* panel = stage_f + (c0 >> 5) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 31) >> 2);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(panel + (((k0 + j) ^ sw) << 4)) = make_float4(vf[4 * j], vf[4 * j + 1], vf[4 * j + 2], vf[4 * j + 3]);
      }
    } else if (row_ok) {
      if (full) {
        if (p.out_bf16 != nullptr) {
          uint4* o = reinterpret_cast<uint4*>(p.out_bf16 + off);
          o[0] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          o[1] = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
        }
        if (p.out_f32 != nullptr) {
          float4* o = reinterpret_cast<float4*>(p.out_f32 + off);
#pragma unroll
          for (int j = 0; j < 4; ++j) o[j] = make_float4(vf[4 * j], vf[4 * j + 1], vf[4 * j + 2], vf[4 * j + 3]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (nb + j >= p.cout) continue;
          if (p.out_bf16 != nullptr) p.out_bf16[off + j] = __float2bfloat16_rn(v[j]);
          if (p.out_f32 != nullptr) p.out_f32[off + j] = vf[j];
        }
      }
    }
  }
  }
  if (p.tma_store) {
    // each epilogue warp stores its own 32-row slab: no cross-warp barrier; TMA clips rows >= M and cols >= Cout
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      const int row0 = (int)(pix0 + q * 32);
      if (p.out_bf16 != nullptr)
        for (int pn = 0; pn * 64 < BLOCK_N && n_blk * BLOCK_N + pn * 64 < p.cout; ++pn)
          tma_store_2d(tmOutB, stage_b + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 64, row0);
      if (p.out_f32 != nullptr)
        for (int pn = 0; pn * 32 < BLOCK_N && n_blk * BLOCK_N + pn * 32 < p.cout; ++pn)
          tma_store_2d(tmOutF, stage_f + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 32, row0);
      if (p.dact != nullptr)
        for (int pn = 0; pn * 64 < BLOCK_N && n_blk * BLOCK_N + pn * 64 < p.cout; ++pn)
          tma_store_2d(tmOutD, stage_d + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 64, row0);
      tma_store_commit();
      if (!DEFER_STORE_WAIT) tma_store_wait_read();       // smem must stay valid until the bulk stores have read it
    }
    __syncwarp();
  }
}

// A warp's 32-row slab of a swizzled staging tile (128-byte panels, 16-byte chunk index XOR (row & 7)) -> global memory with coalesced
// 16-byte stores: consecutive lanes write consecutive chunks of a row (a 128-byte row = 8 lanes = one full line per 8 lanes).  Used instead
// of a TMA store (experiment, off: SIMT_STORE): MEASURED SLOWER than the TMA store it replaces (C64 @32x32: 69.1 vs 53.4 us) although it needs
// no wait for the TMA engine -- kept for the record, the lean epilogue uses staging + TMA store.
template <int ESIZE>     // 2: bf16 panels of 64 columns, 4: fp32 panels of 32 columns
__device__ __forceinline__ void tc_store_slab(const uint8_t* stage_x, void* out, int64_t pix0, int q, int lane, int cout, int col0, int ncols) {
  const int row_chunks = (ncols * ESIZE) >> 4;                   // 16-byte chunks per row of this N block that exist in the tensor
  const int total = 32 * row_chunks;
  uint8_t* obase = reinterpret_cast<uint8_t*>(out) + ((pix0 + q * 32) * (int64_t)cout + col0) * ESIZE;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / row_chunks, cidx = idx - r * row_chunks;
    const int panel = cidx >> 3, k = cidx & 7;
    const uint4 v = *reinterpret_cast<const uint4*>(stage_x + panel * (128 * 128) + (q * 32 + r) * 128 + ((k ^ (r & 7)) << 4));
    *reinterpret_cast<uint4*>(obase + (int64_t)r * cout * ESIZE + cidx * 16) = v;
  }
}

// Lean epilogue for the persistent kernel's hot cases: out = act(acc + bias) with act in {none, SiLU, ReLU}, optional SiLU' tape, bf16 and / or
// fp32 output through the TMA-store staging tile; no add / mul / PReLU.  Every uniform decision is taken ONCE per tile (the generic
// epilogue re-decides per 16-column chunk: ~1000 clk per chunk when the warp has its scheduler to itself, and 140 KB of code), and all
// accumulator columns of the tile (up to 64 at a time) are in flight before the single tcgen05.wait.
__host__ __device__ __forceinline__ bool tc_epilogue_is_lean(const TcParams& p) {
  return p.add == nullptr && p.mul == nullptr && p.act_after_add == 0 && p.tma_store != 0 && p.round_tf32 == 0 &&
         (p.post_act == GA_ACT_NONE || p.post_act == GA_ACT_SILU || p.post_act == GA_ACT_RELU) &&
         (p.dact == nullptr || p.post_act == GA_ACT_SILU);
}

// DIRECT (experiment, off): every thread stores its own output row (128 contiguous bytes for 64 bf16 channels) straight from registers --
// no staging tile, no TMA store, no wait for the TMA engine.  MEASURED SLOWER than staging + TMA store (C64 @32x32, batch 512: 59.7 vs
// 53.4 us): 32 lanes x 16 B to 32 different lines per STG keep the four epilogue warps in the LSU longer than the ~800 clk they wait for
// the bulk store to have read the staging tile.
template <int BLOCK_N, int ACT, bool DACT, bool OUT_B, bool OUT_F, bool CSUM = false, bool DIRECT = false>
__device__ __forceinline__ void tc_epilogue_lean_body(const TcParams& p, uint32_t tmem_acc, int n_blk, uint8_t* stage, const float* s_bias,
                                                      int q, int lane, float* s_csum = nullptr, int64_t pix0 = 0) {
  constexpr int LD = BLOCK_N < 64 ? BLOCK_N : 64;
  const int row = q * 32 + lane;
  uint8_t* stage_b = stage;
  uint8_t* stage_f = stage + (OUT_B ? ((BLOCK_N + 63) / 64) * 16384 : 0);
  uint8_t* stage_d = stage_f + (OUT_F ? (BLOCK_N / 32) * 16384 : 0);
  const uint32_t sw = (uint32_t)(row & 7);
#pragma unroll
  for (int cg = 0; cg < BLOCK_N; cg += LD) {
    uint32_t rr[LD / 16][16];
#pragma unroll
    for (int i = 0; i < LD / 16; ++i) tmem_ld16(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg + i * 16), rr[i]);
    tmem_ld_wait();
#pragma unroll
    for (int ci = 0; ci < LD / 16; ++ci) {
      const int c0 = cg + ci * 16;
      const int nb = n_blk * BLOCK_N + c0;
      if (nb >= p.cout) continue;                               // whole chunk beyond Cout (warp-uniform)
      const int64_t goff = (pix0 + row) * p.cout + nb;          // DIRECT: this thread's row, this chunk's first column
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[ci][j]) + s_bias[c0 + j];
      if (ACT == GA_ACT_SILU) {
        if (DACT) {
          float dv[16];
          silu_with_grad_fast_n<16>(v, v, dv);
          if (DIRECT) {
            uint4* o = reinterpret_cast<uint4*>(p.dact + goff);
            if (nb + 8 <= p.cout) o[0] = make_uint4(pack_bf16x2(dv[0], dv[1]), pack_bf16x2(dv[2], dv[3]), pack_bf16x2(dv[4], dv[5]), pack_bf16x2(dv[6], dv[7]));
            if (nb + 16 <= p.cout) o[1] = make_uint4(pack_bf16x2(dv[8], dv[9]), pack_bf16x2(dv[10], dv[11]), pack_bf16x2(dv[12], dv[13]), pack_bf16x2(dv[14], dv[15]));
          } else {
          uint8_t* panel = stage_d + (c0 >> 6) * (128 * 128) + row * 128;
          const uint32_t k0 = (uint32_t)((c0 & 63) >> 3);
          *reinterpret_cast<uint4*>(panel + (((k0) ^ sw) << 4)) =
              make_uint4(pack_bf16x2(dv[0], dv[1]), pack_bf16x2(dv[2], dv[3]), pack_bf16x2(dv[4], dv[5]), pack_bf16x2(dv[6], dv[7]));
          *reinterpret_cast<uint4*>(panel + (((k0 + 1) ^ sw) << 4)) =
              make_uint4(pack_bf16x2(dv[8], dv[9]), pack_bf16x2(dv[10], dv[11]), pack_bf16x2(dv[12], dv[13]), pack_bf16x2(dv[14], dv[15]));
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = silu_fast(v[j]);
        }
      } else if (ACT == GA_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.0f);
      }
      if (OUT_B && DIRECT) {
        uint4* o = reinterpret_cast<uint4*>(p.out_bf16 + goff);
        if (nb + 8 <= p.cout) o[0] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        if (nb + 16 <= p.cout) o[1] = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
      } else if (OUT_B) {
        uint8_t* panel = stage_b + (c0 >> 6) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 63) >> 3);
        *reinterpret_cast<uint4*>(panel + (((k0) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        *reinterpret_cast<uint4*>(panel + (((k0 + 1) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
      }
      if (OUT_F && DIRECT) {
        float4* o = reinterpret_cast<float4*>(p.out_f32 + goff);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (nb + 4 * j + 4 <= p.cout) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      } else if (OUT_F) {
        uint8_t* panel = stage_f + (c0 >> 5) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 31) >> 2);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(panel + (((k0 + j) ^ sw) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
      if (CSUM) {
        // column sums over this warp's 32 rows of the values AS STORED (bf16-rounded), by recursive halving: after the exchanges over lane
        // bits 4, 3, 2, 1 every lane holds ONE column -- column (lane >> 1) & 15 -- summed over 16 lanes; the last exchange adds the other 16
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __bfloat162float(__float2bfloat16_rn(v[j]));
        float w8[8], w4[4], w2[2];
        const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
        for (int j = 0; j < 8; ++j) w8[j] = (b4 ? v[8 + j] : v[j]) + __shfl_xor_sync(0xffffffffu, b4 ? v[j] : v[8 + j], 16);
#pragma unroll
        for (int j = 0; j < 4; ++j) w4[j] = (b3 ? w8[4 + j] : w8[j]) + __shfl_xor_sync(0xffffffffu, b3 ? w8[j] : w8[4 + j], 8);
#pragma unroll
        for (int j = 0; j < 2; ++j) w2[j] = (b2 ? w4[2 + j] : w4[j]) + __shfl_xor_sync(0xffffffffu, b2 ? w4[j] : w4[2 + j], 4);
        float w1 = (b1 ? w2[1] : w2[0]) + __shfl_xor_sync(0xffffffffu, b1 ? w2[0] : w2[1], 2);
        w1 += __shfl_xor_sync(0xffffffffu, w1, 1);
        if ((lane & 1) == 0) s_csum[q * BLOCK_N + c0 + ((lane >> 1) & 15)] = w1;
      }
    }
  }
}

// -> issues the bulk stores of this warp's 32-row slab and commits them; the CALLER waits (cp.async.bulk.wait_group.read) before the slab is
// written again.  Same staging layout and store boxes as tc_epilogue_tile.
template <int BLOCK_N, bool DIRECT = false, bool SIMT_STORE = false>
__device__ __forceinline__ void tc_epilogue_lean(const TcParams& p, const CUtensorMap* tmOutB, const CUtensorMap* tmOutF,
                                                 const CUtensorMap* tmOutD, uint32_t tmem_acc, int n_blk, int64_t pix0, uint8_t* stage,
                                                 const float* s_bias, int q, int lane, float* s_csum = nullptr) {
  const bool ob = p.out_bf16 != nullptr, of = p.out_f32 != nullptr;
#define GA_LEAN(ACT_, DACT_, OB_, OF_, CS_) tc_epilogue_lean_body<BLOCK_N, ACT_, DACT_, OB_, OF_, CS_, DIRECT>(p, tmem_acc, n_blk, stage, s_bias, q, lane, s_csum, pix0)
  if (p.csum != nullptr) {
    // SE squeeze fused into the conv (host guarantees: no activation, bf16 output only): per-warp column sums -> shared memory ->
    // the 4 epilogue warps meet at a named barrier -> fixed-order sum of the 4 slabs -> [image][128-pixel slice][channel]
    GA_LEAN(GA_ACT_NONE, false, true, false, true);
    asm volatile("bar.sync 2, 128;" ::: "memory");
    const int t = q * 32 + lane;
    if (t < BLOCK_N && n_blk * BLOCK_N + t < p.cout)
      p.csum[(pix0 >> 7) * p.cout + n_blk * BLOCK_N + t] = (s_csum[t] + s_csum[BLOCK_N + t]) + (s_csum[2 * BLOCK_N + t] + s_csum[3 * BLOCK_N + t]);
  } else if (p.post_act == GA_ACT_SILU) {
    if (p.dact != nullptr) {
      if (of) GA_LEAN(GA_ACT_SILU, true, true, true, false);      // (bf16 + fp32 + tape; the engines never ask for fp32 + tape alone)
      else GA_LEAN(GA_ACT_SILU, true, true, false, false);
    } else if (ob && of) GA_LEAN(GA_ACT_SILU, false, true, true, false);
    else if (ob) GA_LEAN(GA_ACT_SILU, false, true, false, false);
    else GA_LEAN(GA_ACT_SILU, false, false, true, false);
  } else if (p.post_act == GA_ACT_RELU) {
    if (ob && of) GA_LEAN(GA_ACT_RELU, false, true, true, false);
    else if (ob) GA_LEAN(GA_ACT_RELU, false, true, false, false);
    else GA_LEAN(GA_ACT_RELU, false, false, true, false);
  } else {
    if (ob && of) GA_LEAN(GA_ACT_NONE, false, true, true, false);
    else if (ob) GA_LEAN(GA_ACT_NONE, false, true, false, false);
    else GA_LEAN(GA_ACT_NONE, false, false, true, false);
  }
#undef GA_LEAN
  if (DIRECT) return;
  uint8_t* stage_b = stage;
  uint8_t* stage_f = stage + (ob ? ((BLOCK_N + 63) / 64) * 16384 : 0);
  uint8_t* stage_d = stage_f + (of ? (BLOCK_N / 32) * 16384 : 0);
  if (SIMT_STORE) {
    __syncwarp();
    const int col0 = n_blk * BLOCK_N;
    const int ncols = (p.cout - col0) < BLOCK_N ? (p.cout - col0) : BLOCK_N;
    if (ob) tc_store_slab<2>(stage_b, p.out_bf16, pix0, q, lane, p.cout, col0, ncols);
    if (of) tc_store_slab<4>(stage_f, p.out_f32, pix0, q, lane, p.cout, col0, ncols);
    if (p.dact != nullptr) tc_store_slab<2>(stage_d, p.dact, pix0, q, lane, p.cout, col0, ncols);
    __syncwarp();
    return;
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    const int row0 = (int)(pix0 + q * 32);
    if (ob)
      for (int pn = 0; pn * 64 < BLOCK_N && n_blk * BLOCK_N + pn * 64 < p.cout; ++pn)
        tma_store_2d(tmOutB, stage_b + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 64, row0);
    if (of)
      for (int pn = 0; pn * 32 < BLOCK_N && n_blk * BLOCK_N + pn * 32 < p.cout; ++pn)
        tma_store_2d(tmOutF, stage_f + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 32, row0);
    if (p.dact != nullptr)
      for (int pn = 0; pn * 64 < BLOCK_N && n_blk * BLOCK_N + pn * 64 < p.cout; ++pn)
        tma_store_2d(tmOutD, stage_d + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 64, row0);
    tma_store_commit();
  }
  __syncwarp();
}

// Lean epilogue with the backward-pass extras: out = (act(acc + bias) + add) * f(mul), add / mul tensors of the output's shape in fp32 or
// bf16; f(mul) is one of the ga_mul_mode factors (PReLU: s_slope holds this N block's slopes).  Each thread owns one output row: its add / mul values of the whole 64-column group are fetched with 16-byte loads BEFORE the
// tcgen05.wait, so the global-load latency overlaps the TMEM round trip (the generic epilogue loads them per 16-column chunk, after the math).
__host__ __device__ __forceinline__ bool tc_epilogue_is_lean_am(const TcParams& p) {
  return (p.add != nullptr || p.mul != nullptr) && p.act_after_add == 0 && p.tma_store != 0 && p.round_tf32 == 0 && p.dact == nullptr &&
         p.post_act != GA_ACT_PRELU && (p.cout % 16) == 0;
}

template <int BLOCK_N>
__device__ __forceinline__ void tc_epilogue_lean_am(const TcParams& p, const CUtensorMap* tmOutB, const CUtensorMap* tmOutF, uint32_t tmem_acc,
                                                    int n_blk, int64_t pix0, uint8_t* stage, const float* s_bias, const float* s_slope,
                                                    int q, int lane) {
  constexpr int LD = BLOCK_N < 64 ? BLOCK_N : 64;
  const int row = q * 32 + lane;
  const int64_t pix = pix0 + row;
  const bool ob = p.out_bf16 != nullptr, of = p.out_f32 != nullptr;
  const bool has_add = p.add != nullptr, add_f32 = p.add_dtype == GA_F32;
  const bool has_mul = p.mul != nullptr, mul_f32 = p.mul_dtype == GA_F32;
  uint8_t* stage_b = stage;
  uint8_t* stage_f = stage + (ob ? ((BLOCK_N + 63) / 64) * 16384 : 0);
  const uint32_t sw = (uint32_t)(row & 7);
#pragma unroll 1
  for (int cg = 0; cg < BLOCK_N; cg += LD) {
    const int nb0 = n_blk * BLOCK_N + cg;
    if (nb0 >= p.cout) break;
    uint32_t rr[LD / 16][16];
#pragma unroll
    for (int i = 0; i < LD / 16; ++i) tmem_ld16(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg + i * 16), rr[i]);
    // columns of this group that exist (cout is a multiple of 16): nv 16-column chunks
    const int nv = (p.cout - nb0) >= LD ? LD / 16 : (p.cout - nb0) / 16;
    uint4 abuf[LD / 4], mbuf[LD / 4];                         // raw add / mul values: fp32 fills LD/4 vectors, bf16 the first LD/8
    const int64_t off = pix * p.cout + nb0;
    const bool row_ok = pix < p.M;                            // ragged last tile of the per-tap kernel: rows past M are never loaded (TMA clips their stores)
#pragma unroll
    for (int i = 0; i < LD / 4; ++i) { abuf[i] = make_uint4(0u, 0u, 0u, 0u); mbuf[i] = make_uint4(0u, 0u, 0u, 0u); }
    if (has_add && row_ok) {
      if (add_f32) {
        const uint4* a4 = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.add) + off);
#pragma unroll
        for (int i = 0; i < LD / 4; ++i) if (i < nv * 4) abuf[i] = __ldg(a4 + i);
      } else {
        const uint4* a4 = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.add) + off);
#pragma unroll
        for (int i = 0; i < LD / 8; ++i) if (i < nv * 2) abuf[i] = __ldg(a4 + i);
      }
    }
    if (has_mul && row_ok) {
      if (mul_f32) {
        const uint4* m4 = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.mul) + off);
#pragma unroll
        for (int i = 0; i < LD / 4; ++i) if (i < nv * 4) mbuf[i] = __ldg(m4 + i);
      } else {
        const uint4* m4 = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.mul) + off);
#pragma unroll
        for (int i = 0; i < LD / 8; ++i) if (i < nv * 2) mbuf[i] = __ldg(m4 + i);
      }
    }
    tmem_ld_wait();
#pragma unroll
    for (int ci = 0; ci < LD / 16; ++ci) {
      if (ci >= nv) break;
      const int c0 = cg + ci * 16;
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[ci][j]) + s_bias[c0 + j];
      apply_act_fast_n<16>(v, p.post_act);
      if (has_add) {
        if (add_f32) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 t = abuf[ci * 4 + j];
            v[4 * j] += __uint_as_float(t.x); v[4 * j + 1] += __uint_as_float(t.y); v[4 * j + 2] += __uint_as_float(t.z); v[4 * j + 3] += __uint_as_float(t.w);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint4 t = abuf[ci * 2 + j];
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) { v[8 * j + 2 * k] += __uint_as_float(w[k] << 16); v[8 * j + 2 * k + 1] += __uint_as_float(w[k] & 0xffff0000u); }
          }
        }
      }
      if (has_mul) {
        float mv[16];
        if (mul_f32) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 t = mbuf[ci * 4 + j];
            mv[4 * j] = __uint_as_float(t.x); mv[4 * j + 1] = __uint_as_float(t.y); mv[4 * j + 2] = __uint_as_float(t.z); mv[4 * j + 3] = __uint_as_float(t.w);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint4 t = mbuf[ci * 2 + j];
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) { mv[8 * j + 2 * k] = __uint_as_float(w[k] << 16); mv[8 * j + 2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u); }
          }
        }
        if (p.mul_mode == GA_MUL_RELU_MASK) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = mv[j] > 0.0f ? v[j] : 0.0f;
        } else if (p.mul_mode == GA_MUL_ELU_FROM_Y) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] *= (mv[j] > 0.0f ? 1.0f : mv[j] + 1.0f);
        } else if (p.mul_mode == GA_MUL_PRELU_FROM_Y) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] *= (mv[j] > 0.0f ? 1.0f : s_slope[c0 + j]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] *= mv[j];
        }
      }
      if (ob) {
        uint8_t* panel = stage_b + (c0 >> 6) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 63) >> 3);
        *reinterpret_cast<uint4*>(panel + (((k0) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        *reinterpret_cast<uint4*>(panel + (((k0 + 1) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
      }
      if (of) {
        uint8_t* panel = stage_f + (c0 >> 5) * (128 * 128) + row * 128;
        const uint32_t k0 = (uint32_t)((c0 & 31) >> 2);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(panel + (((k0 + j) ^ sw) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
    }
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    const int row0 = (int)(pix0 + q * 32);
    if (ob)
      for (int pn = 0; pn * 64 < BLOCK_N && n_blk * BLOCK_N + pn * 64 < p.cout; ++pn)
        tma_store_2d(tmOutB, stage_b + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 64, row0);
    if (of)
      for (int pn = 0; pn * 32 < BLOCK_N && n_blk * BLOCK_N + pn * 32 < p.cout; ++pn)
        tma_store_2d(tmOutF, stage_f + pn * (128 * 128) + q * 32 * 128, n_blk * BLOCK_N + pn * 32, row0);
    tma_store_commit();
  }
  __syncwarp();
}

}  // namespace ga
