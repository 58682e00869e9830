// Fused NVAE decoder cell body for sm_100a:  r = conv1x1_project( SiLU( dwconv5x5( SiLU( conv1x1_expand(x) ) ) ) )
// (/root/reference/src/mlvgms_autoencoders/NVAE/modules/architecture.py:164-173 with the four BatchNorms folded into the three
// convolutions, SURVEY Appendix D).  The 6C-channel hidden tensor never leaves the SM:
//
//   per CTA: one spatial tile of the image batch; the hidden dimension is walked in chunks of 64 channels
//     expand   tcgen05.mma  X[tile px, C] (smem, TMA) x We[chunk, C]^T (smem, TMA)  -> TMEM (double buffered)
//     act      TMEM -> registers, + bias, SiLU, bf16 -> shared memory H (128-byte rows, XOR-swizzled: conflict free)
//     depthwise 5x5 on H out of shared memory: one lane = one channel pair, one warp = a column strip, sliding window in
//              registers, packed FFMA2; + bias, SiLU -> bf16, written straight into the 128B-swizzled K-major layout that
//     project  tcgen05.mma  A2[tile px, chunk] x Wp[Cout, chunk]^T  accumulates into TMEM over all chunks
//   epilogue: TMEM -> + bias -> r (bf16, NHWC) to HBM
//
// HBM traffic per cell drops from (x + 4 x hidden + r) to (x + r): 1.6 GB -> 0.13 GB at 32x32 / batch 512.  The unfused path
// (conv_tc + dwconv5x5_tiled + conv_tc) stays for the taping forward of the attack path and for other shapes.
//
// Warp roles (416 threads): warp 0 = control (TMA producer + MMA issuer, one lane); warps 1-4 = activation (TMEM -> SiLU -> H, and
// the final epilogue), one chunk ahead of warps 5-12 = depthwise (H -> A2): the MUFU-bound and the FMA-bound phases overlap.
// Tiles: 8x8 maps: 2 images / CTA;  16x16: 1 image;  32x32: 8 output rows (+2 halo rows each side, expand recomputed 1.5x).
#include <cuda.h>
#include <stdlib.h>
#include "ga_common.cuh"
#include "tc_ptx.cuh"
#include "tc_host.cuh"

namespace ga {

constexpr int MB_THREADS = 416;      // control warp + 4 activation warps + 8 depthwise warps
#ifndef MB_MAXNREG
#define MB_MAXNREG 128
#endif

template <int W_IMG> struct MbGeom;
template <> struct MbGeom<8>  { static constexpr int IMGS = 2, R_OUT = 8,  HALO = 0, MT_IN = 1, MT_OUT = 1, STRIP_W = 2; };
template <> struct MbGeom<16> { static constexpr int IMGS = 1, R_OUT = 16, HALO = 0, MT_IN = 2, MT_OUT = 2, STRIP_W = 2; };
template <> struct MbGeom<32> { static constexpr int IMGS = 1, R_OUT = 8,  HALO = 2, MT_IN = 3, MT_OUT = 2, STRIP_W = 4; };

struct MbParams {
  int N, H;                     // images, image height (= width = W_IMG)
  int n_tiles;                  // spatial tiles of the batch; CTA b walks tiles b, b + gridDim.x, ... (persistent, one CTA per SM)
  int hidden;                   // 6C (multiple of 64)
  const float* be;              // [hidden] expand bias
  const float* dw_w;            // [hidden/64][25][64] depthwise taps, chunk-major (one 6400-byte bulk copy per chunk)
  const float* dw_b;            // [hidden]
  const float* bp;              // [C] project bias
  __nv_bfloat16* out;           // [N][H][W][C]
  __nv_bfloat16* dact_e;        // TAPE: SiLU'(expand pre-activation), [N][H][W][hidden] (what the attack path's backward multiplies by)
  __nv_bfloat16* dact_dw;       // TAPE: SiLU'(depthwise pre-activation), [N][H][W][hidden]
  // BWD (input gradient of the cell, same pipeline with transposed weights and flipped taps): the two stages multiply by the tapes instead of
  // applying bias + SiLU, and the epilogue is  out_f32 = acc + add_f32
  const __nv_bfloat16* mul_act; // [N][H][W][hidden] factor of the first stage (dact_dw: the gradient enters through the project conv)
  const __nv_bfloat16* mul_dw;  // [N][H][W][hidden] factor of the depthwise stage (dact_e)
  const float* add_f32;         // [N][H][W][C] or NULL: gradient arriving through the skip connection
  float* out_f32;               // [N][H][W][C]
  float* csum;                  // optional: SE squeeze of `out` -- per-image channel sums in the 128-pixel slices of ga_channel_sum, [N][HW/128 or 1][C]
  int act_hi;                   // 1: activation warps are warps 9-12 (scheduler priority is highest-warp-id-first), depthwise warps 1-8
  int sleep_ns;                 // back-off of the SIMT mbarrier polls
  unsigned long long* trace;    // debug (ga_debug_mbconv_trace): clock64 stamps [cta < 8][warp 13][chunk 24][event 8]
};

// mbarrier wait for the SIMT warps: back off between polls so that a waiting warp does not take issue slots from the warps of the
// other role that share its scheduler (activation and depthwise warps wait for each other by design)
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns = 100) {
  uint32_t done;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  while (!done) {
    __nanosleep(ns);
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void simt_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
// 1-D bulk copy global -> shared, completion on an mbarrier (TMA without a tensor map)
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
constexpr int DWW_BYTES = 25 * 64 * 4;
// explicit shared-space accesses on 32-bit addresses: the tile pointers are derived from an aligned-up integer, so the compiler cannot
// prove the address space and would emit generic LD/ST with 64-bit address arithmetic (measured: 2x the integer instructions + spills)
__device__ __forceinline__ uint32_t lds_b32(uint32_t a) { uint32_t v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ float2 lds_f2(uint32_t a) { float2 v; asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ void sts_b32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
// fp16 pair helpers of the F16 depthwise variant (HFMA2 issues one warp-instruction per clock and sub-partition, FFMA2 one per two)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) { uint32_t d; asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo)); return d; }
__device__ __forceinline__ uint32_t hfma2(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ float2 h2_to_f2(uint32_t v) {
  float2 r;
  asm("{\n.reg .f16 l, h;\nmov.b32 {l, h}, %2;\ncvt.f32.f16 %0, l;\ncvt.f32.f16 %1, h;\n}\n" : "=f"(r.x), "=f"(r.y) : "r"(v));
  return r;
}
__device__ __forceinline__ float2 bf2_to_f2(uint32_t v) { return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u)); }

// (a 112-register build -- room for a 256-thread elementwise CTA of another stream beside this CTA -- was tried: registers are per SM sub-partition
// and 4 of this CTA's 13 warps share one, so the second CTA does not fit anyway; DESIGN.md)
template <int C, int W_IMG, int NBUF, bool TRACE = false, bool F16 = false, bool TAPE = false, bool BWD = false>
__global__ void __maxnreg__(MB_MAXNREG) mbconv_fused_kernel(const __grid_constant__ CUtensorMap tmX,
                                                                     const __grid_constant__ CUtensorMap tmWe,
                                                                     const __grid_constant__ CUtensorMap tmWp, const MbParams p) {
  using G = MbGeom<W_IMG>;
  constexpr int KB = C / 64;                           // 64-channel K blocks of the expand GEMM
  constexpr int R_IN = G::R_OUT + 2 * G::HALO;
  constexpr int X_BYTES = G::MT_IN * KB * 16384;
  constexpr int WE_BYTES = KB * 8192;                  // one chunk: 64 hidden rows x C
  constexpr int WP_BYTES = C * 128;                    // one chunk: C rows x 64 hidden
  constexpr int H_BYTES = G::MT_IN * 16384;
  constexpr int A2_BYTES = G::MT_OUT * 16384;
  constexpr uint32_t EXP_COLS = G::MT_IN * 64;         // one expand accumulator buffer
  constexpr uint32_t PROJ_OFF = 2 * EXP_COLS;
  static_assert(PROJ_OFF + G::MT_OUT * C <= 512, "TMEM budget");
  static_assert(G::IMGS * R_IN * W_IMG == G::MT_IN * 128 && G::IMGS * G::R_OUT * W_IMG == G::MT_OUT * 128, "tile geometry");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* hdr = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(hdr);
  uint64_t* x_full = bars + 0;
  uint64_t* we_full = bars + 1;          // [2]
  uint64_t* we_empty = bars + 3;         // [2]
  uint64_t* wp_full = bars + 5;          // [2]
  uint64_t* wp_empty = bars + 7;         // [2]
  uint64_t* exp_full = bars + 9;         // [2]
  uint64_t* exp_empty = bars + 11;       // [2]
  uint64_t* a2_full = bars + 13;
  uint64_t* a2_empty = bars + 14;
  uint64_t* proj_full = bars + 15;
  uint64_t* dww_full = bars + 16;        // [2]
  uint64_t* h_full = bars + 18;          // [2]
  uint64_t* h_empty = bars + 20;         // [2]
  uint64_t* x_free = bars + 22;          // all expand MMAs of a tile have read X: the next tile may be loaded
  uint64_t* proj_empty = bars + 23;      // the epilogue has drained the project accumulator
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 24);
  uint8_t* sX = hdr + 1024;
  uint8_t* sWe = sX + X_BYTES;
  uint8_t* sWp = sWe + NBUF * WE_BYTES;
  uint8_t* sH = sWp + NBUF * WP_BYTES;
  uint8_t* sA2 = sH + 2 * H_BYTES;                                   // H is double buffered (activation warps run one chunk ahead)
  float* s_dww = reinterpret_cast<float*>(sA2 + A2_BYTES);          // [2][25][64] depthwise taps of the current / next chunk
  float* s_be = s_dww + 2 * 25 * 64;
  float* s_bp = s_be + p.hidden;                                    // [C] project bias (the depthwise bias is read through L1: 2 floats per lane and chunk)
  float* s_cs = s_bp + C;                                           // [2][4][64] per-warp column sums of the epilogue (double buffered)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nch = p.hidden / 64;
  // persistent: this CTA's tiles, and ONE chunk counter g over all of them (chunk k of local tile i is g = i * nch + k).  Every ring
  // (weights, expand accumulator, H, A2, taps) is indexed by g, so the next tile's first chunks are loaded / expanded / activated while
  // the depthwise warps finish this tile and the activation warps drain its project accumulator: no per-tile head or tail.
  const int my_tiles = ((int)p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int g_total = my_tiles * nch;
  // debug timeline: lane 0 of every warp stamps clock64 at the role's synchronisation points (traced CTAs: the first 4 and 4 of a later wave)
  const int tr_cta = TRACE ? (blockIdx.x < 4 ? (int)blockIdx.x : ((blockIdx.x >= 1184 && blockIdx.x < 1188) ? (int)blockIdx.x - 1180 : -1)) : -1;
  auto stamp = [&](int k, int ev) {
    if (TRACE && tr_cta >= 0 && (threadIdx.x & 31) == 0 && k < 24)
      p.trace[((size_t)(tr_cta * 13 + (threadIdx.x >> 5)) * 24 + k) * 8 + ev] = (unsigned long long)clock64();
  };
  stamp(0, 7);

  // ---- local tile i -> (first image, first output row)
  auto tile_origin = [&](int i, int& n0, int& y0) {
    const int t = (int)blockIdx.x + i * (int)gridDim.x;
    if (W_IMG == 8) { n0 = t * 2; y0 = 0; }
    else if (W_IMG == 16) { n0 = t; y0 = 0; }
    else { n0 = t / (W_IMG / G::R_OUT); y0 = (t % (W_IMG / G::R_OUT)) * G::R_OUT; }
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX); tma_prefetch_desc(&tmWe); tma_prefetch_desc(&tmWp);
    mbar_init(x_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&we_full[i], 1); mbar_init(&we_empty[i], 1); mbar_init(&wp_full[i], 1); mbar_init(&wp_empty[i], 1);
      mbar_init(&exp_full[i], 1); mbar_init(&exp_empty[i], 4); mbar_init(&dww_full[i], 1);
      mbar_init(&h_full[i], 4); mbar_init(&h_empty[i], 8);
    }
    mbar_init(a2_full, 8); mbar_init(a2_empty, 1); mbar_init(proj_full, 1);      // a2_full: one arrival per depthwise warp
    mbar_init(x_free, 1); mbar_init(proj_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    // expand bias pre-halved: SiLU(v) = h + h tanh(h) with h = v/2 = fma(acc, 0.5, be/2) -- exact (power-of-two scaling), one FMA-pipe op less
    if (!BWD) {
      for (int i = threadIdx.x - 32; i < p.hidden; i += MB_THREADS - 32) s_be[i] = 0.5f * p.be[i];
      for (int i = threadIdx.x - 32; i < C; i += MB_THREADS - 32) s_bp[i] = p.bp[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ======================================================================= control: TMA producer + MMA issuer
    if (elect_one_sync()) {      // (elected lane, not `lane == 0`: uniform-datapath instructions then issue without an elect / branch loop each)
      constexpr uint32_t idesc_e = make_idesc(128, 64);
      constexpr uint32_t idesc_p = make_idesc(128, C);
      auto load_we = [&](int gj) {
        const int b = gj % NBUF, j = gj % nch;
        mbar_expect_tx(&we_full[b], WE_BYTES);
        for (int kb = 0; kb < KB; ++kb) tma_load_2d(&tmWe, &we_full[b], sWe + b * WE_BYTES + kb * 8192, kb * 64, j * 64);
      };
      auto load_dww = [&](int gj) {
        mbar_expect_tx(&dww_full[gj & 1], DWW_BYTES);
        bulk_load_1d(s_dww + (gj & 1) * 25 * 64, p.dw_w + (size_t)(gj % nch) * 25 * 64, DWW_BYTES, &dww_full[gj & 1]);
      };
      auto load_wp = [&](int gj) {
        const int b = gj % NBUF, j = gj % nch;
        mbar_expect_tx(&wp_full[b], WP_BYTES);
        tma_load_2d(&tmWp, &wp_full[b], sWp + b * WP_BYTES, j * 64, 0);
      };
      auto load_x = [&](int i) {
        int n0, y0;
        tile_origin(i, n0, y0);
        mbar_expect_tx(x_full, X_BYTES);
        for (int m = 0; m < G::MT_IN; ++m)
          for (int kb = 0; kb < KB; ++kb) {
            uint8_t* dst = sX + (m * KB + kb) * 16384;
            if (W_IMG == 8) tma_load_4d(&tmX, x_full, dst, kb * 64, 0, 0, n0);
            else tma_load_4d(&tmX, x_full, dst, kb * 64, 0, y0 - G::HALO + m * (128 / W_IMG), n0);
          }
      };
      auto expand = [&](int g) {
        if (g >= 1) {                                     // lazy refill of the buffer expand(g-1) has finished with
          const int gj = g - 1 + NBUF;
          if (gj < g_total) { mbar_wait(&we_empty[(g - 1) % NBUF], ((g - 1) / NBUF) & 1); load_we(gj); }
        }
        const int i = g / nch, k = g - i * nch;
        if (k == 0) { mbar_wait(x_full, i & 1); if (i == 0) stamp(0, 6); }
        mbar_wait(&we_full[g % NBUF], (g / NBUF) & 1);
        if (g >= 2) mbar_wait(&exp_empty[g & 1], ((g - 2) >> 1) & 1);
        tc_fence_after();
        const uint32_t we_addr = smem_u32(sWe + (g % NBUF) * WE_BYTES);
        for (int m = 0; m < G::MT_IN; ++m) {
          const uint32_t d = tmem_base + (g & 1) * EXP_COLS + m * 64;
          for (int kb = 0; kb < KB; ++kb) {
            const uint32_t a_addr = smem_u32(sX + (m * KB + kb) * 16384);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16(d, make_smem_desc(a_addr + kk * 32), make_smem_desc(we_addr + kb * 8192 + kk * 32), idesc_e, (kb > 0 || kk > 0) ? 1u : 0u);
          }
        }
        umma_commit(&exp_full[g & 1]);
        umma_commit(&we_empty[g % NBUF]);
        stamp(g, 0);
        if (k == nch - 1 && i + 1 < my_tiles) {           // the tile's last expand: X is free once these MMAs have run -> prefetch the next tile
          umma_commit(x_free);
          mbar_wait(x_free, i & 1);
          load_x(i + 1);
        }
      };
      auto project = [&](int g) {
        if (g >= 1) {
          const int gj = g - 1 + NBUF;
          if (gj < g_total) { mbar_wait(&wp_empty[(g - 1) % NBUF], ((g - 1) / NBUF) & 1); load_wp(gj); }
        }
        stamp(g, 1);
        mbar_wait(a2_full, g & 1);
        stamp(g, 2);
        if (g + 2 < g_total) load_dww(g + 2);             // every SIMT thread has taken chunk g's taps into registers
        mbar_wait(&wp_full[g % NBUF], (g / NBUF) & 1);
        const int i = g / nch, k = g - i * nch;
        if (k == 0 && i >= 1) mbar_wait(proj_empty, (i - 1) & 1);      // the previous tile's accumulator has been read out
        tc_fence_after();
        const uint32_t wp_addr = smem_u32(sWp + (g % NBUF) * WP_BYTES);
        for (int m = 0; m < G::MT_OUT; ++m) {
          const uint32_t a_addr = smem_u32(sA2 + m * 16384);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16(tmem_base + PROJ_OFF + m * C, make_smem_desc(a_addr + kk * 32), make_smem_desc(wp_addr + kk * 32), idesc_p,
                      (k > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(a2_empty);
        umma_commit(&wp_empty[g % NBUF]);
        stamp(g, 3);
        if (k == nch - 1) umma_commit(proj_full);
      };
      // ---- prologue: the first activation tile and the first weight chunks
      load_x(0);
      for (int j = 0; j < NBUF && j < g_total; ++j) { load_we(j); load_wp(j); }
      for (int j = 0; j < 2 && j < g_total; ++j) load_dww(j);
      expand(0);
      for (int g = 0; g < g_total; ++g) {
        if (g + 1 < g_total) expand(g + 1);
        project(g);
      }
    }
    __syncwarp();
  } else if (p.act_hi ? warp >= 9 : warp <= 4) {
    // ======================================================================= activation warps (1-4, one per TMEM lane quadrant):
    // expand accumulator -> + bias -> SiLU -> bf16 -> H[k & 1] (swizzled rows), one chunk ahead of the depthwise warps
    const int q = warp & 3;                  // TMEM lane quadrant this warp may read
    int cs_batch = 0;                        // channel-sum batches done (selects the shared-memory buffer)
    // ---- project accumulator of local tile j -> + bias -> r (bf16) -> HBM
    auto epilogue = [&](int j) {
      int n0, y0;
      tile_origin(j, n0, y0);
      stamp(j, 4);
      mbar_wait_backoff(proj_full, j & 1, (uint32_t)p.sleep_ns);
      stamp(j, 5);
      tc_fence_after();
      const int64_t pix0 = (W_IMG == 32) ? ((int64_t)n0 * p.H + y0) * W_IMG : (int64_t)n0 * p.H * W_IMG;
      const int64_t total_pix = (int64_t)p.N * p.H * W_IMG;
#pragma unroll 1
      for (int m = 0; m < G::MT_OUT; ++m) {
        const int64_t pix = pix0 + m * 128 + q * 32 + lane;
        // 64 accumulator columns in flight per tcgen05.wait (the round trip is ~1k clk for a lone warp; C / 16 of them in a row were 10% of
        // the CTA's lifetime), then one full 128-byte line per thread
        if (BWD) {
          // out_f32 = acc + add_f32: 32 columns per step (the skip gradient's 128 bytes are in flight while the accumulator is read)
          const bool row_ok = pix < total_pix;
#pragma unroll 1
          for (int c0 = 0; c0 < C; c0 += 32) {
            float4 av[8];
            if (p.add_f32 != nullptr && row_ok) {
              const float4* ap = reinterpret_cast<const float4*>(p.add_f32 + pix * C + c0);
#pragma unroll
              for (int i = 0; i < 8; ++i) av[i] = __ldg(ap + i);
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) av[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            uint32_t r[2][16];
#pragma unroll
            for (int c16 = 0; c16 < 2; ++c16) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + PROJ_OFF + m * C + c0 + c16 * 16, r[c16]);
            tmem_ld_wait();
            if (m == G::MT_OUT - 1 && c0 + 32 >= C) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(proj_empty);
            }
            if (row_ok) {
              float4* o = reinterpret_cast<float4*>(p.out_f32 + pix * C + c0);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const uint32_t* rr = &r[i >> 2][(i & 3) * 4];
                o[i] = make_float4(__uint_as_float(rr[0]) + av[i].x, __uint_as_float(rr[1]) + av[i].y, __uint_as_float(rr[2]) + av[i].z,
                                   __uint_as_float(rr[3]) + av[i].w);
              }
            }
          }
          continue;
        }
#pragma unroll 1
        for (int c0 = 0; c0 < C; c0 += 64) {
          uint32_t r[4][16];
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + PROJ_OFF + m * C + c0 + c16 * 16, r[c16]);
          tmem_ld_wait();
          if (m == G::MT_OUT - 1 && c0 + 64 >= C) {       // last read of the accumulator: hand it back before the stores go out
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(proj_empty);
          }
          const bool row_ok = pix < total_pix;
          uint4* o = reinterpret_cast<uint4*>(p.out + pix * C + c0);
          const uint32_t bp_a = smem_u32(s_bp) + c0 * 4;
          float* cs = s_cs + (cs_batch & 1) * 256 + q * 64;
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16) {
            uint32_t pk[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              const float2 b = lds_f2(bp_a + (c16 * 16 + 2 * jj) * 4);
              pk[jj] = pack_bf16x2(__uint_as_float(r[c16][2 * jj]) + b.x, __uint_as_float(r[c16][2 * jj + 1]) + b.y);
            }
            if (row_ok) {
              o[2 * c16] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
              o[2 * c16 + 1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            }
            if (p.csum != nullptr) {
              // column sums over this warp's 32 pixels of the values AS STORED (bf16), by recursive halving (the scheme of the persistent 3x3
              // kernel's epilogue, conv_tc_epilogue.cuh): after the exchanges over lane bits 4..1 a lane holds one column, summed over 16 lanes
              float v[16];
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
                v[2 * jj] = row_ok ? __uint_as_float(pk[jj] << 16) : 0.f;
                v[2 * jj + 1] = row_ok ? __uint_as_float(pk[jj] & 0xffff0000u) : 0.f;
              }
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
              if ((lane & 1) == 0) cs[c16 * 16 + ((lane >> 1) & 15)] = w1;
            }
          }
          if (p.csum != nullptr) {
            // the four activation warps meet (named barrier 2; the buffers alternate, so one barrier per batch is enough), then a fixed-order
            // sum of the four 32-pixel slabs -> [image][128-pixel slice][channel]; 8x8 maps: two images of 64 pixels per accumulator tile
            asm volatile("bar.sync 2, 128;" ::: "memory");
            const float* cb = s_cs + (cs_batch & 1) * 256;
            const int t = q * 32 + lane;
            if (W_IMG == 8) {
              const int img = t >> 6, ch = t & 63;
              if (n0 + img < p.N) p.csum[(int64_t)(n0 + img) * C + c0 + ch] = cb[(2 * img) * 64 + ch] + cb[(2 * img + 1) * 64 + ch];
            } else if (t < 64) {
              p.csum[(((pix0 + m * 128) >> 7)) * C + c0 + t] = (cb[t] + cb[64 + t]) + (cb[128 + t] + cb[192 + t]);
            }
            ++cs_batch;
          }
        }
      }
    };
    int ti = 0, k = 0, n0, y0;
    tile_origin(0, n0, y0);
    const int epi_after = nch > 1 ? 1 : 0;   // the previous tile is drained after this tile's second chunk has been activated (see below)
    for (int g = 0; g < g_total; ++g) {
      stamp(g, 0);
      mbar_wait_backoff(&exp_full[g & 1], (g >> 1) & 1, (uint32_t)p.sleep_ns);
      stamp(g, 1);
      if (g >= 2) mbar_wait_backoff(&h_empty[g & 1], ((g - 2) >> 1) & 1, (uint32_t)p.sleep_ns);          // depthwise(g-2) has read this H buffer
      stamp(g, 2);
      tc_fence_after();
      const uint32_t hb = smem_u32(sH) + (g & 1) * H_BYTES;
      const uint32_t be_a = smem_u32(s_be) + k * 256;
#pragma unroll
      for (int m = 0; m < G::MT_IN; ++m) {
        const int pin = m * 128 + q * 32 + lane;
        bool in_img = true;
        if (G::HALO > 0) {
          const int y = y0 - G::HALO + (pin / W_IMG) % R_IN;
          in_img = y >= 0 && y < p.H;                     // halo rows outside the image are the conv's zero padding
        }
        const uint32_t row = hb + pin * 128;
        // TAPE: the global pixel this thread's row belongs to (halo rows of a 32x32 tile belong to the neighbouring tiles)
        bool own = false;
        int64_t gpix = 0;
        uint4 mv[8];                 // BWD: this pixel's 64 tape factors of the chunk (in flight while the accumulator is read)
        if (BWD) {
          if (W_IMG == 32) {
            own = in_img;            // every row of the tile inside the image, halo rows included
            gpix = (((int64_t)n0 * p.H + y0 - G::HALO + (pin >> 5)) << 5) + (pin & 31);
          } else {
            gpix = (int64_t)n0 * p.H * W_IMG + pin;
            own = gpix < (int64_t)p.N * p.H * W_IMG;
          }
          const uint4* mp = reinterpret_cast<const uint4*>(p.mul_act + gpix * p.hidden + k * 64);
#pragma unroll
          for (int i = 0; i < 8; ++i) mv[i] = own ? __ldg(mp + i) : make_uint4(0u, 0u, 0u, 0u);
        }
        if (TAPE) {
          if (W_IMG == 32) {
            const int rt = (pin >> 5) - G::HALO;
            own = rt >= 0 && rt < G::R_OUT;
            gpix = (((int64_t)n0 * p.H + y0 + rt) << 5) + (pin & 31);
          } else {
            gpix = (int64_t)n0 * p.H * W_IMG + pin;
            own = gpix < (int64_t)p.N * p.H * W_IMG;
          }
        }
        // all 64 columns of this lane's pixel in flight before ONE wait: a tcgen05.ld round trip costs ~1k cycles, and one warp per
        // scheduler cannot hide it behind anything else
        uint32_t r[4][16];
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16)
          tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (g & 1) * EXP_COLS + m * 64 + c16 * 16, r[c16]);
        tmem_ld_wait();
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16) {
          uint32_t pk[8], dk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (BWD) {               // gradient through the first GEMM times the tape; rows outside the image are the conv's zero padding
              const uint4 mq = mv[c16 * 2 + (j >> 2)];
              const uint32_t mw = (j & 3) == 0 ? mq.x : ((j & 3) == 1 ? mq.y : ((j & 3) == 2 ? mq.z : mq.w));
              const float2 f = bf2_to_f2(mw);
              pk[j] = own ? pack_bf16x2(__uint_as_float(r[c16][2 * j]) * f.x, __uint_as_float(r[c16][2 * j + 1]) * f.y) : 0u;
              continue;
            }
            const float2 b = lds_f2(be_a + (c16 * 16 + 2 * j) * 4);
            const float h0 = fmaf(__uint_as_float(r[c16][2 * j]), 0.5f, b.x), h1 = fmaf(__uint_as_float(r[c16][2 * j + 1]), 0.5f, b.y);
            const float t0 = tanh_approx(h0), t1 = tanh_approx(h1);
            const float v0 = fmaf(h0, t0, h0), v1 = fmaf(h1, t1, h1);
            // TAPE: SiLU' from the same tanh (act_grad_fast_n's form: 1/2 + (t + h (1 - t^2)) / 2)
            if (TAPE) dk[j] = pack_bf16x2(fmaf(0.5f, fmaf(h0, fmaf(-t0, t0, 1.0f), t0), 0.5f), fmaf(0.5f, fmaf(h1, fmaf(-t1, t1, 1.0f), t1), 0.5f));
            // fp16 H: SiLU(h) >= -0.28, so only the upper end can leave the fp16 range -- clamp instead of producing inf
            pk[j] = in_img ? (F16 ? pack_f16x2(fminf(v0, 60000.f), fminf(v1, 60000.f)) : pack_bf16x2(v0, v1)) : 0u;
          }
          const uint32_t ch0 = (uint32_t)(c16 * 2);                       // 16-byte chunk index inside the 128-byte row
          sts_v4(row + (((ch0) ^ (pin & 7)) << 4), pk[0], pk[1], pk[2], pk[3]);
          sts_v4(row + (((ch0 + 1) ^ (pin & 7)) << 4), pk[4], pk[5], pk[6], pk[7]);
          if (TAPE && own) {
            uint4* o = reinterpret_cast<uint4*>(p.dact_e + gpix * p.hidden + k * 64 + c16 * 16);
            o[0] = make_uint4(dk[0], dk[1], dk[2], dk[3]);
            o[1] = make_uint4(dk[4], dk[5], dk[6], dk[7]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&exp_empty[g & 1]); mbar_arrive(&h_full[g & 1]); }
      stamp(g, 3);
      // the previous tile's accumulator completes about when the depthwise warps start on this tile's first chunk; by then this warp has
      // produced the chunk after it, so draining now keeps the depthwise warps fed (activation first, epilogue second)
      if (ti >= 1 && k == epi_after) epilogue(ti - 1);
      if (++k == nch) { k = 0; ++ti; tile_origin(ti, n0, y0); }
    }
    if (my_tiles > 0) epilogue(my_tiles - 1);
  } else {
    // ======================================================================= depthwise warps (5-12): 5x5 + bias + SiLU: H -> A2
    const int sw = p.act_hi ? warp - 1 : warp - 5;   // 0..7
    // strip of this warp
    const int img = (W_IMG == 8) ? (sw >> 2) : 0;
    const int cs = (W_IMG == 8) ? (sw & 3) * G::STRIP_W : sw * G::STRIP_W;
    // per-column shared-memory addresses of this lane's channel pair: pixel p = (row)*W + x sits in 128-byte row p, its 16-byte chunk
    // j at (j ^ (p & 7)); W is a multiple of 8, so p & 7 == x & 7 and only the row term changes inside the loops
    const uint32_t lch = (uint32_t)(lane >> 2), lof = (uint32_t)(lane & 3) * 4;
    uint32_t h_col[G::STRIP_W + 4];
    bool col_ok[G::STRIP_W + 4];
    uint32_t a2_col[G::STRIP_W];
#pragma unroll
    for (int c = 0; c < G::STRIP_W + 4; ++c) {
      const int x = cs - 2 + c;
      col_ok[c] = x >= 0 && x < W_IMG;
      h_col[c] = (uint32_t)((img * R_IN * W_IMG + x) * 128) + ((lch ^ (uint32_t)(x & 7)) << 4) + lof;
    }
#pragma unroll
    for (int c = 0; c < G::STRIP_W; ++c)
      a2_col[c] = smem_u32(sA2) + (img * G::R_OUT * W_IMG + cs + c) * 128 + ((lch ^ (uint32_t)((cs + c) & 7)) << 4) + lof;
    if constexpr (F16) {
      // fp16 variant: H holds fp16 pairs, the 25 taps and the accumulators are fp16 pairs (one register each), so a whole strip (all R_OUT rows)
      // accumulates in ONE pass -- no input row is read twice -- and the 25 multiply-adds per output pair are 25 HFMA2 instead of 25 FFMA2
      // (half the fp32-pipe cycles) with no unpack.  The 25-term fp16 accumulation adds ~1e-3 relative rounding noise, about half of what the
      // bf16 rounding of the result adds anyway; the bias, SiLU and the bf16 rounding stay fp32.
      int ti_d = 0, n0d = 0, y0d = 0;
      if (TAPE) tile_origin(0, n0d, y0d);
      for (int g = 0, kc = 0; g < g_total; ++g, kc = (kc + 1 == nch) ? 0 : kc + 1) {
        uint32_t wt[25];
        stamp(g, 0);
        mbar_wait_backoff(&dww_full[g & 1], (g >> 1) & 1, (uint32_t)p.sleep_ns);
        {
          const uint32_t wsrc = smem_u32(s_dww) + ((g & 1) * 25 * 64 + 2 * lane) * 4;
#pragma unroll
          for (int t = 0; t < 25; ++t) { const float2 w = lds_f2(wsrc + t * 256); wt[t] = pack_f16x2(w.x, w.y); }
        }
        const float2 b2 = __ldg(reinterpret_cast<const float2*>(p.dw_b + kc * 64 + 2 * lane));
        stamp(g, 1);
        mbar_wait_backoff(&h_full[g & 1], (g >> 1) & 1, (uint32_t)p.sleep_ns);
        stamp(g, 2);
        const uint32_t hb = smem_u32(sH) + (g & 1) * H_BYTES;
        constexpr int RP = G::R_OUT;
        uint32_t acc[RP][G::STRIP_W];
#pragma unroll
        for (int oy = 0; oy < RP; ++oy)
#pragma unroll
          for (int c = 0; c < G::STRIP_W; ++c) acc[oy][c] = 0u;
#pragma unroll
        for (int ir = 0; ir < RP + 4; ++ir) {
          const int iy = G::HALO - 2 + ir;
          if (iy < 0 || iy >= R_IN) continue;
          uint32_t in[G::STRIP_W + 4];
#pragma unroll
          for (int c = 0; c < G::STRIP_W + 4; ++c) {
            in[c] = 0u;
            if (col_ok[c]) in[c] = lds_b32(hb + h_col[c] + iy * (W_IMG * 128));
          }
#pragma unroll
          for (int ky = 0; ky < 5; ++ky) {
            const int oy = ir - ky;
            if (oy < 0 || oy >= RP) continue;
#pragma unroll
            for (int c = 0; c < G::STRIP_W; ++c)
#pragma unroll
              for (int kx = 0; kx < 5; ++kx) acc[oy][c] = hfma2(wt[ky * 5 + kx], in[c + kx], acc[oy][c]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_empty[g & 1]);
        stamp(g, 3);
        if (g >= 1) mbar_wait_backoff(a2_empty, (g - 1) & 1, (uint32_t)p.sleep_ns);
        stamp(g, 4);
#pragma unroll
        for (int oy = 0; oy < RP; ++oy)
#pragma unroll
          for (int c = 0; c < G::STRIP_W; ++c) {
            const float2 a = h2_to_f2(acc[oy][c]);
            if (TAPE) {
              // SiLU and SiLU' from one tanh each; the derivative goes to the tape of the attack path's backward (coalesced: a warp's 32
              // channel pairs are 128 contiguous bytes of the pixel's hidden row)
              const float h0 = 0.5f * (a.x + b2.x), h1 = 0.5f * (a.y + b2.y);
              const float t0 = tanh_approx(h0), t1 = tanh_approx(h1);
              sts_b32(a2_col[c] + oy * (W_IMG * 128), pack_bf16x2(fmaf(h0, t0, h0), fmaf(h1, t1, h1)));
              int64_t gpix;
              bool ok = true;
              if (W_IMG == 32) gpix = (((int64_t)n0d * p.H + y0d + oy) << 5) + cs + c;
              else if (W_IMG == 16) gpix = (int64_t)n0d * 256 + oy * 16 + cs + c;
              else { gpix = (int64_t)(n0d + img) * 64 + oy * 8 + cs + c; ok = n0d + img < p.N; }
              if (ok)
                *reinterpret_cast<uint32_t*>(p.dact_dw + gpix * p.hidden + kc * 64 + 2 * lane) =
                    pack_bf16x2(fmaf(0.5f, fmaf(h0, fmaf(-t0, t0, 1.0f), t0), 0.5f), fmaf(0.5f, fmaf(h1, fmaf(-t1, t1, 1.0f), t1), 0.5f));
            } else {
              sts_b32(a2_col[c] + oy * (W_IMG * 128), pack_bf16x2(silu_fast(a.x + b2.x), silu_fast(a.y + b2.y)));
            }
          }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(a2_full);
        stamp(g, 5);
        if (TAPE && kc + 1 == nch) { ++ti_d; tile_origin(ti_d, n0d, y0d); }
      }
    } else {
    int ti_b = 0, n0b = 0, y0b = 0;
    if (BWD) tile_origin(0, n0b, y0b);
    for (int g = 0, kc = 0; g < g_total; ++g, kc = (kc + 1 == nch) ? 0 : kc + 1) {
      float2 wt[25];
      {
        stamp(g, 0);
        mbar_wait_backoff(&dww_full[g & 1], (g >> 1) & 1, (uint32_t)p.sleep_ns);
        const uint32_t wsrc = smem_u32(s_dww) + ((g & 1) * 25 * 64 + 2 * lane) * 4;
#pragma unroll
        for (int t = 0; t < 25; ++t) wt[t] = lds_f2(wsrc + t * 256);
      }
      const float2 b2 = BWD ? make_float2(0.f, 0.f) : __ldg(reinterpret_cast<const float2*>(p.dw_b + kc * 64 + 2 * lane));
      // BWD: this lane's tape word of output (0, 0) of the warp's strip; output (oy, c) is (oy * W + c) pixels further.  The lines the store
      // phases will read are pulled into L2 now.
      const char* tape0 = nullptr;
      bool tape_ok = true;
      const uint32_t pstride = (uint32_t)p.hidden * 2u;
      if (BWD) {
        int64_t gp0;
        if (W_IMG == 32) gp0 = (((int64_t)n0b * p.H + y0b) << 5) + cs;
        else if (W_IMG == 16) gp0 = (int64_t)n0b * 256 + cs;
        else { gp0 = (int64_t)(n0b + img) * 64 + cs; tape_ok = n0b + img < p.N; }
        tape0 = reinterpret_cast<const char*>(p.mul_dw + gp0 * p.hidden + kc * 64 + 2 * lane);
        if (tape_ok) {
#pragma unroll
          for (int oy = 0; oy < G::R_OUT; ++oy)
#pragma unroll
            for (int c = 0; c < G::STRIP_W; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(tape0 + (uint32_t)(oy * W_IMG + c) * pstride));
        }
      }
      stamp(g, 1);
      mbar_wait_backoff(&h_full[g & 1], (g >> 1) & 1, (uint32_t)p.sleep_ns);
      stamp(g, 2);
      const uint32_t hb = smem_u32(sH) + (g & 1) * H_BYTES;
      // the strip's rows are produced in passes of RP rows (RP + 4 input rows each): RP x STRIP_W accumulators + 25 taps stay in
      // registers under the 128-register cap of a 13-warp CTA (16K registers per SM sub-partition, 4 warps on one of them)
      constexpr int RP = (G::R_OUT * G::STRIP_W > 16) ? G::R_OUT / 2 : G::R_OUT;
#pragma unroll
      for (int pass = 0; pass < G::R_OUT / RP; ++pass) {
        if (BWD && pass > 0 && W_IMG != 16) {         // (measured per shape: 32x32 769 -> 663 us, 8x8 195 -> 178 us; 16x16 is faster without: 331 vs 354 us)
          // BWD: the taps are re-read from shared memory for every pass, so their 50 registers are free while the previous pass' store phase
          // keeps all its tape loads in flight (with the taps live the compiler serialised them: 2.8k clk per store phase)
          const uint32_t wsrc = smem_u32(s_dww) + ((g & 1) * 25 * 64 + 2 * lane) * 4;
#pragma unroll
          for (int t = 0; t < 25; ++t) wt[t] = lds_f2(wsrc + t * 256);
        }
        float2 acc[RP][G::STRIP_W];
#pragma unroll
        for (int oy = 0; oy < RP; ++oy)
#pragma unroll
          for (int c = 0; c < G::STRIP_W; ++c) acc[oy][c] = b2;
#pragma unroll
        for (int ir = 0; ir < RP + 4; ++ir) {
          const int iy = pass * RP + G::HALO - 2 + ir;     // input row (H-tile coordinates) feeding this pass
          if (iy < 0 || iy >= R_IN) continue;             // above / below the tile: zero rows (whole-image tiles only)
          float2 in[G::STRIP_W + 4];
#pragma unroll
          for (int c = 0; c < G::STRIP_W + 4; ++c) {
            in[c] = make_float2(0.f, 0.f);
            if (col_ok[c])
              in[c] = bf2_to_f2(lds_b32(hb + h_col[c] + iy * (W_IMG * 128)));
          }
#pragma unroll
          for (int ky = 0; ky < 5; ++ky) {
            const int oy = ir - ky;                       // output row (inside the pass) fed by input row ir through tap row ky
            if (oy < 0 || oy >= RP) continue;
#pragma unroll
            for (int c = 0; c < G::STRIP_W; ++c)
#pragma unroll
              for (int kx = 0; kx < 5; ++kx) acc[oy][c] = ffma2(wt[ky * 5 + kx], in[c + kx], acc[oy][c]);
          }
        }
        if (pass == G::R_OUT / RP - 1) {
          __syncwarp();
          if (lane == 0) mbar_arrive(&h_empty[g & 1]);                     // this warp is done reading H[g & 1]
        }
        if (pass == 0) stamp(g, 3);
        if (pass == 0 && g >= 1) mbar_wait_backoff(a2_empty, (g - 1) & 1, (uint32_t)p.sleep_ns); // project(k-1) has consumed A2
        if (pass == 0) stamp(g, 4);
        if (BWD) {
          uint32_t dv[RP][G::STRIP_W];
#pragma unroll
          for (int oy = 0; oy < RP; ++oy)
#pragma unroll
            for (int c = 0; c < G::STRIP_W; ++c)
              dv[oy][c] = tape_ok ? __ldg(reinterpret_cast<const uint32_t*>(tape0 + (uint32_t)((pass * RP + oy) * W_IMG + c) * pstride)) : 0u;
#pragma unroll
          for (int oy = 0; oy < RP; ++oy)
#pragma unroll
            for (int c = 0; c < G::STRIP_W; ++c) {
              const float2 f = bf2_to_f2(dv[oy][c]);
              sts_b32(a2_col[c] + (pass * RP + oy) * (W_IMG * 128), pack_bf16x2(acc[oy][c].x * f.x, acc[oy][c].y * f.y));
            }
        } else {
#pragma unroll
        for (int oy = 0; oy < RP; ++oy)
#pragma unroll
          for (int c = 0; c < G::STRIP_W; ++c)
            sts_b32(a2_col[c] + (pass * RP + oy) * (W_IMG * 128), pack_bf16x2(silu_fast(acc[oy][c].x), silu_fast(acc[oy][c].y)));
        }
      }
      fence_proxy_async_smem();                                            // generic-proxy writes -> visible to the MMA (async proxy)
      __syncwarp();
      // every depthwise warp arrives on its own (count 8): no warp waits for the slowest one at a CTA barrier, it goes on to the next
      // chunk's taps / H tile and only meets the others again at a2_empty, after its next pass-0 accumulation (ncu: 13% barrier stalls)
      if (lane == 0) mbar_arrive(a2_full);
      stamp(g, 5);
      if (BWD && kc + 1 == nch) { ++ti_b; tile_origin(ti_b, n0b, y0b); }
    }
    }
  }
  stamp(1, 7);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

// ----------------------------------------------------------------------------- host side
typedef CUresult (*PFN_mbEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_mbEncodeTiled mb_encode_fn() {
  static PFN_mbEncodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_mbEncodeTiled>(ptr);
  }
  return fn;
}

static int mb_encode_2d(CUtensorMap* tm, const void* base, int cols, int rows, int box_rows) {
  PFN_mbEncodeTiled enc = mb_encode_fn();
  GA_CHECK(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  GA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(weights %d x %d, box rows %d) failed: %d", rows, cols, box_rows, (int)r);
  return 0;
}

static int mb_encode_x(CUtensorMap* tm, const ga_tensor* t, int bw, int bh, int bn) {
  PFN_mbEncodeTiled enc = mb_encode_fn();
  GA_CHECK(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[4] = {(cuuint64_t)t->c, (cuuint64_t)t->w, (cuuint64_t)t->h, (cuuint64_t)t->n};
  cuuint64_t strides[3] = {(cuuint64_t)t->c * 2, (cuuint64_t)t->w * t->c * 2, (cuuint64_t)t->h * t->w * t->c * 2};
  cuuint32_t box[4] = {64u, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, t->data, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  GA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(activation n=%d h=%d w=%d c=%d) failed: %d", t->n, t->h, t->w, t->c, (int)r);
  return 0;
}

static unsigned long long* g_mb_trace = nullptr;

template <int C, int W_IMG, int NBUF, bool TRACE = false, bool F16 = false, bool TAPE = false, bool BWD = false>
static int launch_mbconv(const ga_tensor* x, const void* we, const void* wp, const MbParams& p, cudaStream_t s) {
  using G = MbGeom<W_IMG>;
  constexpr int KB = C / 64;
  const int smem = 1024 /*align*/ + 1024 /*header*/ + G::MT_IN * KB * 16384 + NBUF * (KB * 8192 + C * 128) + 2 * G::MT_IN * 16384 +
                   G::MT_OUT * 16384 + 2 * DWW_BYTES + p.hidden * 4 + C * 4 + 2 * 4 * 64 * 4;
  GA_CHECK(smem <= 227 * 1024, "ga_mbconv_fused: shared memory request %d too large", smem);
  static int configured = 0;
  if (configured < smem) {
    GA_CUDA(cudaFuncSetAttribute(mbconv_fused_kernel<C, W_IMG, NBUF, TRACE, F16, TAPE, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  CUtensorMap tmX, tmWe, tmWp;
  if (W_IMG == 8) { if (mb_encode_x(&tmX, x, 8, 8, 2)) return 1; }
  else if (mb_encode_x(&tmX, x, W_IMG, 128 / W_IMG, 1)) return 1;
  if (mb_encode_2d(&tmWe, we, C, p.hidden, 64)) return 1;          // [hidden][C]: box = 64 hidden rows x 64 k
  if (mb_encode_2d(&tmWp, wp, p.hidden, C, C)) return 1;           // [C][hidden]: box = C rows x 64 k
  int tiles;
  if (W_IMG == 8) tiles = (x->n + 1) / 2;
  else if (W_IMG == 16) tiles = x->n;
  else tiles = x->n * (W_IMG / G::R_OUT);
  MbParams q = p;
  q.n_tiles = tiles;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  mbconv_fused_kernel<C, W_IMG, NBUF, TRACE, F16, TAPE, BWD><<<grid, MB_THREADS, smem, s>>>(tmX, tmWe, tmWp, q);
  GA_LAUNCH_OK();
  return 0;
}

}  // namespace ga

using namespace ga;

extern "C" int ga_mbconv_fused_supported(const ga_tensor* x, int hidden) {
  if (!x || x->dtype != GA_BF16 || x->h != x->w || hidden % 64 != 0 || hidden < 64 || hidden > 1536) return 0;
  if ((((uintptr_t)x->data) & 15) != 0) return 0;
  return (x->w == 8 && x->c == 256) || (x->w == 16 && x->c == 128) || (x->w == 32 && x->c == 64);
}

extern "C" int ga_mbconv_fused_ex(const ga_tensor* x, const void* we_tc, const float* be, const float* dw_w, const float* dw_b,
                                  const void* wp_tc, const float* bp, int hidden, const ga_tensor* out, float* csum_out,
                                  const ga_tensor* dact_e, const ga_tensor* dact_dw, void* stream);

extern "C" int ga_mbconv_fused(const ga_tensor* x, const void* we_tc, const float* be, const float* dw_w, const float* dw_b,
                               const void* wp_tc, const float* bp, int hidden, const ga_tensor* out, void* stream) {
  return ga_mbconv_fused_ex(x, we_tc, be, dw_w, dw_b, wp_tc, bp, hidden, out, nullptr, nullptr, nullptr, stream);
}

extern "C" int ga_mbconv_fused_ex(const ga_tensor* x, const void* we_tc, const float* be, const float* dw_w, const float* dw_b,
                                  const void* wp_tc, const float* bp, int hidden, const ga_tensor* out, float* csum_out,
                                  const ga_tensor* dact_e, const ga_tensor* dact_dw, void* stream) {
  GA_CHECK(x && we_tc && be && dw_w && dw_b && wp_tc && bp && out, "ga_mbconv_fused: null argument");
  GA_CHECK(ga_mbconv_fused_supported(x, hidden), "ga_mbconv_fused: unsupported problem (n=%d h=%d w=%d c=%d hidden=%d)", x->n, x->h, x->w,
           x->c, hidden);
  GA_CHECK(out->dtype == GA_BF16 && same_shape(x, out), "ga_mbconv_fused: output must be bf16 with the input's shape");
  GA_CHECK(((((uintptr_t)we_tc) | ((uintptr_t)wp_tc) | ((uintptr_t)out->data)) & 15) == 0, "ga_mbconv_fused: pointers must be 16-byte aligned");
  if (numel(x) == 0) return 0;
  MbParams p;
  p.N = x->n; p.H = x->h; p.hidden = hidden; p.be = be; p.dw_w = dw_w; p.dw_b = dw_b; p.bp = bp;
  p.out = (__nv_bfloat16*)out->data;
  p.csum = csum_out;
  GA_CHECK((dact_e == nullptr) == (dact_dw == nullptr), "ga_mbconv_fused: the two tape tensors go together");
  const bool tape = dact_e != nullptr;
  if (tape) {
    GA_CHECK(dact_e->dtype == GA_BF16 && dact_dw->dtype == GA_BF16 && dact_e->n == x->n && dact_e->h == x->h && dact_e->w == x->w && dact_e->c == hidden &&
                 same_shape(dact_e, dact_dw), "ga_mbconv_fused: tape tensors must be bf16 [n][h][w][hidden]");
    GA_CHECK(((((uintptr_t)dact_e->data) | ((uintptr_t)dact_dw->data)) & 15) == 0, "ga_mbconv_fused: tape pointers must be 16-byte aligned");
  }
  p.dact_e = tape ? (__nv_bfloat16*)dact_e->data : nullptr;
  p.dact_dw = tape ? (__nv_bfloat16*)dact_dw->data : nullptr;
  static int act_hi = -1, sleep_ns = -1;
  if (act_hi < 0) { const char* e = getenv("GA_MB_ACT_HI"); act_hi = e ? atoi(e) : 0; }
  if (sleep_ns < 0) { const char* e = getenv("GA_MB_SLEEP_NS"); sleep_ns = e ? atoi(e) : 100; }
  p.act_hi = act_hi; p.sleep_ns = sleep_ns; p.trace = g_mb_trace;
  cudaStream_t s = (cudaStream_t)stream;
  // GA_MB_F16 (default 1): fp16 hidden tile + HFMA2 depthwise accumulation (one pass per strip, no bf16 unpack; more accurate than the bf16
  // hidden tile as long as |hidden| and the 25-tap sums stay inside the fp16 range, which the clamp at 6e4 and BN-folded NVAE weights give);
  // 0: bf16 hidden tile, fp32 FFMA2 accumulation (bit-identical to the three separate kernels)
  static int f16 = -1;
  if (f16 < 0) { const char* e = getenv("GA_MB_F16"); f16 = e ? atoi(e) : 1; }
  if (tape) {          // the taping variant exists for the fp16 hidden tile only
    if (x->w == 8) return launch_mbconv<256, 8, 1, false, true, true>(x, we_tc, wp_tc, p, s);
    if (x->w == 16) return launch_mbconv<128, 16, 1, false, true, true>(x, we_tc, wp_tc, p, s);
    return launch_mbconv<64, 32, 2, false, true, true>(x, we_tc, wp_tc, p, s);
  }
  if (f16) {
    if (x->w == 8) return launch_mbconv<256, 8, 1, false, true>(x, we_tc, wp_tc, p, s);
    if (x->w == 16) return launch_mbconv<128, 16, 1, false, true>(x, we_tc, wp_tc, p, s);
    if (p.trace != nullptr) return launch_mbconv<64, 32, 2, true, true>(x, we_tc, wp_tc, p, s);
    static int nbuf32 = -1;
    if (nbuf32 < 0) { const char* e = getenv("GA_MB_NBUF32"); nbuf32 = e ? atoi(e) : 2; }
    if (nbuf32 == 1) return launch_mbconv<64, 32, 1, false, true>(x, we_tc, wp_tc, p, s);
    return launch_mbconv<64, 32, 2, false, true>(x, we_tc, wp_tc, p, s);
  }
  if (x->w == 8) return launch_mbconv<256, 8, 1>(x, we_tc, wp_tc, p, s);
  if (x->w == 16) return launch_mbconv<128, 16, 1>(x, we_tc, wp_tc, p, s);
  if (p.trace != nullptr) return launch_mbconv<64, 32, 2, true>(x, we_tc, wp_tc, p, s);
  return launch_mbconv<64, 32, 2>(x, we_tc, wp_tc, p, s);
}

// Input gradient of the decoder cell in one kernel (the attack path's backward; architecture.py:164-173 under torch.autograd.grad, untargeted.py:146,201):
//   out = add + expand^T( dact_e * dw5x5^T( dact_dw * project^T(g) ) )
// = the forward pipeline with the two 1x1 convs swapped and transposed (wpT_tc [hidden][C] feeds the first GEMM, weT_tc [C][hidden] the second), the taps
// flipped (dw_wT, chunk-major), the tapes of ga_mbconv_fused_ex as stage factors, no biases, bf16 hidden tile with fp32 accumulation (gradients need the
// bf16 exponent range), fp32 result.
extern "C" int ga_mbconv_fused_bwd(const ga_tensor* g, const void* wpT_tc, const float* dw_wT, const ga_tensor* dact_dw, const ga_tensor* dact_e,
                                   const void* weT_tc, const ga_tensor* add, int hidden, const ga_tensor* out, void* stream) {
  GA_CHECK(g && wpT_tc && dw_wT && dact_dw && dact_e && weT_tc && out, "ga_mbconv_fused_bwd: null argument");
  GA_CHECK(ga_mbconv_fused_supported(g, hidden), "ga_mbconv_fused_bwd: unsupported problem (n=%d h=%d w=%d c=%d hidden=%d)", g->n, g->h, g->w, g->c, hidden);
  GA_CHECK(out->dtype == GA_F32 && same_shape(g, out) && (!add || (add->dtype == GA_F32 && same_shape(g, add))),
           "ga_mbconv_fused_bwd: out (and add) must be fp32 with the gradient's shape");
  GA_CHECK(dact_e->dtype == GA_BF16 && dact_dw->dtype == GA_BF16 && dact_e->n == g->n && dact_e->h == g->h && dact_e->w == g->w && dact_e->c == hidden &&
               same_shape(dact_e, dact_dw), "ga_mbconv_fused_bwd: tape tensors must be bf16 [n][h][w][hidden]");
  GA_CHECK(((((uintptr_t)wpT_tc) | ((uintptr_t)weT_tc) | ((uintptr_t)out->data) | ((uintptr_t)dact_e->data) | ((uintptr_t)dact_dw->data) |
             (add ? (uintptr_t)add->data : 0)) & 15) == 0, "ga_mbconv_fused_bwd: pointers must be 16-byte aligned");
  if (numel(g) == 0) return 0;
  MbParams p;
  memset(&p, 0, sizeof(p));
  p.N = g->n; p.H = g->h; p.hidden = hidden; p.dw_w = dw_wT;
  p.mul_act = (const __nv_bfloat16*)dact_dw->data; p.mul_dw = (const __nv_bfloat16*)dact_e->data;
  p.add_f32 = add ? (const float*)add->data : nullptr; p.out_f32 = (float*)out->data;
  p.sleep_ns = 100;
  cudaStream_t s = (cudaStream_t)stream;
  if (g->w == 8) return launch_mbconv<256, 8, 1, false, false, false, true>(g, wpT_tc, weT_tc, p, s);
  if (g->w == 16) return launch_mbconv<128, 16, 1, false, false, false, true>(g, wpT_tc, weT_tc, p, s);
  p.trace = g_mb_trace;
  if (p.trace != nullptr) return launch_mbconv<64, 32, 2, true, false, false, true>(g, wpT_tc, weT_tc, p, s);
  return launch_mbconv<64, 32, 2, false, false, false, true>(g, wpT_tc, weT_tc, p, s);
}

// debug: per-role clock64 timeline of the 32x32 fused cell (scripts/trace_mbconv.py); buf = device uint64[8 * 13 * 24 * 8] or NULL (off)
extern "C" int ga_debug_mbconv_trace(unsigned long long* buf) {
  ga::g_mb_trace = buf;
  return 0;
}
