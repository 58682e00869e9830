// tcgen05 / TMEM / TMA implicit-GEMM convolution for sm_100a (bf16 operands, fp32 accumulation in TMEM).
//
// Replaces the cuDNN convolutions behind the NVAE residual cells, samplers and combiners
// (/root/reference/src/mlvgms_autoencoders/NVAE/modules/architecture.py:96-218, NVAE/model.py:184-231,310-313)
// and the VGG11 body / head GEMMs (src/classifier/model.py:31-50) on the bf16 product path.
//
// GEMM view   D[M = pixels, N = Cout] = A[M, K] * B[N, K]^T,   K = taps * Cin (+ Cin2 of a second 1x1 source)
//   * A is never materialised: one CTA owns 128 output pixels laid out as a (bn x bh x bw) box of the NHWC
//     activation tensor; for every filter tap the TMA engine fetches the box shifted by (ky-pad, kx-pad) with
//     hardware zero fill outside the image -- that IS the zero padding of the convolution (im2col by TMA).
//   * B (weights, [Cout][K] K-major bf16) streams through the same mbarrier ring.
//   * 64-channel K blocks land in shared memory in the 128-byte-swizzled K-major layout that tcgen05.mma
//     consumes directly (UMMA descriptors, SBO = 1024 B); 4 MMAs (K=16 each) per block, issued by ONE thread.
//   * The fp32 accumulator tile (128 lanes x BLOCK_N columns) lives in tensor memory; 4 epilogue warps read it
//     back with tcgen05.ld (one pixel row per thread), fuse bias + activation + residual add and store bf16/fp32.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 = epilogue.
// One output tile per CTA; 2 CTAs are co-resident per SM (<= 97 KB smem, <= 256 TMEM columns each) so one CTA's
// epilogue overlaps the other's main loop.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include "ga_common.cuh"
#include "tc_ptx.cuh"
#include "conv_tc_epilogue.cuh"
#include "tc_host.cuh"

namespace ga {

constexpr int TC_BLOCK_M = 128;
constexpr int TC_BLOCK_K = 64;                       // bf16 elements = 128 bytes = one swizzle row
constexpr int TC_A_STAGE_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;   // 16 KB
constexpr int TC_THREADS = 192;


template <int BLOCK_N, int STAGES, bool GENERAL_ACT>
__global__ void __launch_bounds__(TC_THREADS, BLOCK_N <= 64 ? 5 : (BLOCK_N == 128 ? 4 : 2)) conv_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                             const __grid_constant__ CUtensorMap tmA2,
                                                             const __grid_constant__ CUtensorMap tmB,
                                                             const __grid_constant__ CUtensorMap tmOutB,
                                                             const __grid_constant__ CUtensorMap tmOutF,
                                                             const __grid_constant__ CUtensorMap tmOutD, const TcParams p) {
  constexpr int B_STAGE_BYTES = BLOCK_N * TC_BLOCK_K * 2;
  constexpr int STAGE_BYTES = TC_A_STAGE_BYTES + B_STAGE_BYTES;
  constexpr uint32_t TMEM_COLS = BLOCK_N < 32 ? 32 : BLOCK_N;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: swizzle-128B atoms (8 rows x 128 B) must start on a 1024 B boundary
  // (aligned up by indexing the __shared__ array, not through an integer cast: the compiler keeps the shared address space and emits
  // LDS / STS with 32-bit addresses instead of generic LD / ST with 64-bit address arithmetic)
  uint8_t* smem_hdr = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int HDR_BYTES = GENERAL_ACT ? 4096 : 2048;
  uint8_t* smem = smem_hdr + HDR_BYTES;              // operand ring / epilogue staging (1024-aligned)
  uint8_t* smem_a = smem;
  // 32-channel K blocks use half-size stages (more co-resident CTAs for the small-channel, high-resolution layers)
  const int a_stride = p.k32 ? TC_A_STAGE_BYTES / 2 : TC_A_STAGE_BYTES;
  const int b_stride = p.k32 ? B_STAGE_BYTES / 2 : B_STAGE_BYTES;
  uint8_t* smem_b = smem + STAGES * a_stride;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_hdr);   // header: barriers, TMEM address; bias tile after the ring
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  float* s_slope = reinterpret_cast<float*>(smem_hdr + 128 + 1024);
  float* s_bias = reinterpret_cast<float*>(smem_hdr + 128);      // header (4 KB): 128 B of barriers + up to 1 KB of bias + up to 1 KB of PReLU slopes

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // 1-D grid, N block fastest: the CTAs that share an A tile (same pixels, different output-channel blocks) are scheduled back to back, so
  // the tile is fetched from HBM once and hits L2 afterwards (ncu, 1x1 expand 64 -> 384: the A tensor was read 3x from DRAM)
  const int n_blk = blockIdx.x % p.n_blocks;

  // ---- tile -> pixel box
  int n0, y0, x0;
  {
    const int t = blockIdx.x / p.n_blocks;
    if (p.bn > 1) { n0 = t * p.bn; y0 = 0; x0 = 0; }
    else {
      const int per_img = p.tiles_x * p.tiles_y;
      n0 = t / per_img;
      const int rem = t - n0 * per_img;
      y0 = (rem / p.tiles_x) * p.bh;
      x0 = (rem % p.tiles_x) * p.bw;
    }
  }
  const int64_t pix0 = ((int64_t)n0 * p.H + y0) * p.W + x0;
  const int num_kb = p.taps * p.kc1 + p.kc2;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.kc2 > 0) tma_prefetch_desc(&tmA2);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // whole warp allocates tensor memory
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================================================================== TMA producer
    int stage = 0; uint32_t phase = 0;
    const int bk = (p.k32 || p.tf32) ? 32 : TC_BLOCK_K;
    for (int kb = 0; kb < num_kb; ++kb) {
      if (elect_one_sync()) {      // (not `lane == 0`: see tc_ptx.cuh -- uniform-datapath instructions issue directly under an elected lane)
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_expect_tx(&full_bar[stage], p.k32 ? STAGE_BYTES / 2 : STAGE_BYTES);
        uint8_t* a_dst = smem_a + stage * a_stride;
        uint8_t* b_dst = smem_b + stage * b_stride;
        int kcoord;
        if (kb < p.taps * p.kc1) {
          const int tap = kb / p.kc1, cc = kb - tap * p.kc1;
          const int ky = tap / p.kw, kx = tap - ky * p.kw;
          tma_load_4d(&tmA, &full_bar[stage], a_dst, cc * bk, x0 * p.stride + kx - p.pad, y0 * p.stride + ky - p.pad, n0);
          kcoord = tap * p.cin + cc * bk;
        } else {
          const int cc = kb - p.taps * p.kc1;
          tma_load_4d(&tmA2, &full_bar[stage], a_dst, cc * bk, x0, y0, n0);
          kcoord = p.taps * p.cin + cc * bk;
        }
        tma_load_2d(&tmB, &full_bar[stage], b_dst, kcoord, n_blk * BLOCK_N);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    constexpr uint32_t idesc = make_idesc(TC_BLOCK_M, BLOCK_N);
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < num_kb; ++kb) {
      if (elect_one_sync()) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem_a + stage * a_stride);
        const uint32_t b_addr = smem_u32(smem_b + stage * b_stride);
        if (p.tf32) {
          constexpr uint32_t idesc32 = make_idesc_tf32(TC_BLOCK_M, BLOCK_N);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_tf32(tmem_base, make_smem_desc(a_addr + k * 32), make_smem_desc(b_addr + k * 32), idesc32, (kb > 0 || k > 0) ? 1u : 0u);
        } else if (p.k32) {
#pragma unroll
          for (int k = 0; k < 2; ++k)
            umma_bf16(tmem_base, make_smem_desc_sw64(a_addr + k * 32), make_smem_desc_sw64(b_addr + k * 32), idesc, (kb > 0 || k > 0) ? 1u : 0u);
        } else {
#pragma unroll
          for (int k = 0; k < TC_BLOCK_K / 16; ++k)      // K advance inside the swizzle atom: + 32 bytes = + 2 in the descriptor's low word
            umma_bf16(tmem_base, smem_desc_from_lo(smem_desc_lo(a_addr) + k * 2), smem_desc_from_lo(smem_desc_lo(b_addr) + k * 2), idesc,
                      (kb > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty_bar[stage]);                     // smem slot free once these MMAs retire
        if (kb == num_kb - 1) umma_commit(tmem_full_bar);   // accumulator complete
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else {
    // ===================================================================== epilogue (warps 2..5)
    const int et = threadIdx.x - 64;                 // 0..127
    for (int i = et; i < BLOCK_N; i += 128) {
      const int n = n_blk * BLOCK_N + i;
      s_bias[i] = (p.bias != nullptr && n < p.cout) ? p.bias[n] : 0.f;
      if (GENERAL_ACT) s_slope[i] = (p.act_slope != nullptr && n < p.cout) ? p.act_slope[n] : 0.f;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");   // epilogue-only named barrier
    // GENERAL_ACT (compile time): PReLU slopes and/or act(acc + bias + add); the hot NVAE path compiles without it
    const int q = warp & 3;                          // TMEM lane quadrant this warp may access
    if (lane == 0) mbar_wait(tmem_full_bar, 0);
    __syncwarp();
    tc_fence_after();
    // staging tiles for the TMA store re-use the (now idle) operand ring: every MMA has retired, so every TMA load has landed and
    // every operand read is done
    tc_epilogue_tile<BLOCK_N, GENERAL_ACT>(p, &tmOutB, &tmOutF, &tmOutD, tmem_base, n_blk, pix0, p.partial ? (p.H - y0) * p.W : 128, smem,
                                           s_bias, s_slope, q, lane);
  }
  // ---- teardown: every tcgen05 op of this CTA is complete (the epilogue waited for the last commit)
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ----------------------------------------------------------------------------- host side
struct TileGeom { int bw, bh, bn, tiles_x, tiles_y, partial; int64_t m_tiles; };

static bool tile_geometry(int N, int H, int W, TileGeom* g) {
  g->partial = 0;
  if (W >= 128) {
    if (W % 128) return false;
    g->bw = 128; g->bh = 1; g->bn = 1;
  } else {
    if (128 % W) return false;
    g->bw = W;
    const int rows = 128 / W;
    if (H >= rows) { g->bh = rows; g->bn = 1; g->partial = (H % rows) != 0; }      // e.g. 12 x 16 maps: 8-row tiles, the 2nd half empty
    else { if (rows % H) return false; g->bh = H; g->bn = rows / H; }
  }
  g->tiles_x = W / g->bw; g->tiles_y = (H + g->bh - 1) / g->bh;
  g->m_tiles = g->bn > 1 ? (N + g->bn - 1) / g->bn : (int64_t)N * g->tiles_x * g->tiles_y;
  return true;
}

static int encode_act_map(CUtensorMap* tm, const ga_tensor* t, const TileGeom& g, int stride = 1, int block_k = TC_BLOCK_K, int esize = 2) {
  cuuint64_t dims[4] = {(cuuint64_t)t->c, (cuuint64_t)t->w, (cuuint64_t)t->h, (cuuint64_t)t->n};
  cuuint64_t strides[3] = {(cuuint64_t)t->c * esize, (cuuint64_t)t->w * t->c * esize, (cuuint64_t)t->h * t->w * t->c * esize};
  // stride-2 convs: the box spans stride*bw x stride*bh input pixels and the TMA engine keeps every stride-th one
  // (ceil(box/elementStride) elements per dimension land in shared memory)
  cuuint32_t box[4] = {(cuuint32_t)block_k, (cuuint32_t)(g.bw * stride), (cuuint32_t)(g.bh * stride), (cuuint32_t)g.bn};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  return encode_tiled_cached(tm, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, t->data, dims, strides, box,
                             estr, block_k * esize == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
}

static int encode_weight_map(CUtensorMap* tm, const void* w, int cout, int ktot, int block_n, int block_k = TC_BLOCK_K, int esize = 2) {
  cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)cout};
  cuuint64_t strides[1] = {(cuuint64_t)ktot * esize};
  cuuint32_t box[2] = {(cuuint32_t)block_k, (cuuint32_t)block_n};
  cuuint32_t estr[2] = {1, 1};
  return encode_tiled_cached(tm, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w, dims, strides, box, estr,
                             block_k * esize == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

static int encode_out_map(CUtensorMap* tm, void* base, int cout, int64_t m, int esize) {
  cuuint64_t dims[2] = {(cuuint64_t)cout, (cuuint64_t)m};
  cuuint64_t strides[1] = {(cuuint64_t)cout * esize};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esize), 32u};      // one 128-byte panel x one warp's 32 rows
  cuuint32_t estr[2] = {1, 1};
  return encode_tiled_cached(tm, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE);
}

template <int BLOCK_N, int STAGES, bool GENERAL_ACT>
static int launch_tc_(const CUtensorMap& a, const CUtensorMap& a2, const CUtensorMap& b, const CUtensorMap& ob, const CUtensorMap& of,
                     const CUtensorMap& od, const TcParams& p, dim3 grid, cudaStream_t s) {
  constexpr int ring = STAGES * (TC_A_STAGE_BYTES + BLOCK_N * TC_BLOCK_K * 2);
  constexpr int max_staging = 2 * ((BLOCK_N + 63) / 64) * 16384 + (BLOCK_N / 32) * 16384;
  constexpr int HDR_BYTES = GENERAL_ACT ? 4096 : 2048;
  constexpr int max_smem = 1024 /*align*/ + HDR_BYTES + (ring > max_staging ? ring : max_staging);
  static bool configured = false;
  if (!configured) {
    GA_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BLOCK_N, STAGES, GENERAL_ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 max_smem > 227 * 1024 ? 227 * 1024 : max_smem));
    configured = true;
  }
  int staging = 0;
  if (p.tma_store) staging = ((p.out_bf16 ? 1 : 0) + (p.dact ? 1 : 0)) * ((BLOCK_N + 63) / 64) * 16384 + (p.out_f32 ? (BLOCK_N / 32) * 16384 : 0);
  const int ring_rt = p.k32 ? ring / 2 : ring;
  const int smem = 1024 + HDR_BYTES + (ring_rt > staging ? ring_rt : staging);
  GA_CHECK(smem <= 227 * 1024, "conv_tc: shared memory request %d too large", smem);
  conv_tc_kernel<BLOCK_N, STAGES, GENERAL_ACT><<<grid, TC_THREADS, smem, s>>>(a, a2, b, ob, of, od, p);
  GA_LAUNCH_OK();
  return 0;
}

template <int BLOCK_N, int STAGES>
static int launch_tc(const CUtensorMap& a, const CUtensorMap& a2, const CUtensorMap& b, const CUtensorMap& ob, const CUtensorMap& of,
                     const CUtensorMap& od, const TcParams& p, dim3 grid, cudaStream_t s) {
  if (p.act_after_add != 0 || p.post_act == GA_ACT_PRELU || (p.mul != nullptr && p.mul_mode == GA_MUL_PRELU_FROM_Y))
    return launch_tc_<BLOCK_N, STAGES, true>(a, a2, b, ob, of, od, p, grid, s);
  return launch_tc_<BLOCK_N, STAGES, false>(a, a2, b, ob, of, od, p, grid, s);
}

static int pick_block_n(int cout) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("GA_TC_BLOCK_N");
    forced = e ? atoi(e) : 0;
  }
  if (forced == 32 || forced == 64 || forced == 128 || forced == 256) return forced;
  if (cout <= 32) return 32;
  if (cout <= 64) return 64;
  return 128;
}

}  // namespace ga

using namespace ga;

extern "C" int ga_conv2d_tc_supported(const ga_tensor* in, const ga_tensor* in2, const ga_conv_desc* d, int cout) {
  if (!in || !d) return 0;
  if (d->tf32 ? (in->dtype != GA_F32 || in2 != nullptr || in->c % 4 != 0) : (in->dtype != GA_BF16)) return 0;
  if ((d->stride != 1 && d->stride != 2) || d->up != 1 || d->pre_op != GA_PRE_NONE) return 0;
  if (!((d->kh == 1 && d->kw == 1 && d->pad == 0) || (d->kh == 3 && d->kw == 3 && d->pad == 1))) return 0;
  if (in->c % 8 != 0 || cout < 1) return 0;
  if (in2 && (d->stride != 1 || in2->dtype != GA_BF16 || in2->c % 8 != 0 || in2->n != in->n || in2->h != in->h || in2->w != in->w)) return 0;
  TileGeom g;
  const int Ho = (in->h + 2 * d->pad - d->kh) / d->stride + 1, Wo = (in->w + 2 * d->pad - d->kw) / d->stride + 1;
  if (!tile_geometry(in->n, Ho, Wo, &g)) return 0;
  if ((((uintptr_t)in->data) & 15) != 0) return 0;
  return 1;
}

extern "C" int ga_conv2d_tc(const ga_tensor* in, const ga_tensor* in2, const ga_conv_desc* d, const ga_tensor* add,
                            const ga_tensor* out_bf16, const ga_tensor* out_f32, void* stream) {
  GA_CHECK(in && d && (out_bf16 || out_f32), "ga_conv2d_tc: null argument");
  const ga_tensor* out = out_bf16 ? out_bf16 : out_f32;
  GA_CHECK(ga_conv2d_tc_supported(in, in2, d, out->c), "ga_conv2d_tc: unsupported problem (n=%d h=%d w=%d cin=%d k=%d stride=%d pre=%d)",
           in->n, in->h, in->w, in->c, d->kh, d->stride, d->pre_op);
  const int Ho = (in->h + 2 * d->pad - d->kh) / d->stride + 1, Wo = (in->w + 2 * d->pad - d->kw) / d->stride + 1;
  GA_CHECK(out->n == in->n && out->h == Ho && out->w == Wo, "ga_conv2d_tc: output spatial shape mismatch");
  GA_CHECK(!out_bf16 || out_bf16->dtype == GA_BF16, "ga_conv2d_tc: out_bf16 must be bf16");
  GA_CHECK(!out_f32 || out_f32->dtype == GA_F32, "ga_conv2d_tc: out_f32 must be fp32");
  GA_CHECK(!(out_bf16 && out_f32) || same_shape(out_bf16, out_f32), "ga_conv2d_tc: the two outputs differ in shape");
  if (add) GA_CHECK(same_shape(add, out), "ga_conv2d_tc: add shape mismatch");
  const int taps = d->kh * d->kw;
  const int ktot = taps * in->c + (in2 ? in2->c : 0);
  GA_CHECK(d->ktot == ktot, "ga_conv2d_tc: weight row length %d != kh*kw*cin(+cin2) = %d", d->ktot, ktot);
  GA_CHECK((((uintptr_t)d->weight) & 15) == 0, "ga_conv2d_tc: weight pointer must be 16-byte aligned");
  if (numel(out) == 0) return 0;

  TileGeom g;
  tile_geometry(in->n, Ho, Wo, &g);
  const int block_n = pick_block_n(out->c);
  // 32-channel K blocks when Cin is an odd multiple of 32 (32, 96, ...): a 64-channel box would be half empty (zero-filled) for the
  // last block of every tap -- at Cin = 32 that is half of all operand traffic and half of all MMAs
  static int k32_enabled = -1;
  if (k32_enabled < 0) { const char* e = getenv("GA_TC_K32"); k32_enabled = e ? atoi(e) : 1; }
  const int tf32 = d->tf32 ? 1 : 0;
  const int k32 = (!tf32 && k32_enabled && !in2 && (in->c % 64) == 32) ? 1 : 0;
  const int bk = (k32 || tf32) ? 32 : TC_BLOCK_K;
  const int esize = tf32 ? 4 : 2;
  TcParams p;
  p.taps = taps; p.kw = d->kw; p.pad = d->pad; p.stride = d->stride;
  p.k32 = k32; p.tf32 = tf32;
  p.cin = in->c; p.kc1 = (in->c + bk - 1) / bk; p.kc2 = in2 ? (in2->c + TC_BLOCK_K - 1) / TC_BLOCK_K : 0;
  p.bw = g.bw; p.bh = g.bh; p.bn = g.bn; p.tiles_x = g.tiles_x; p.tiles_y = g.tiles_y;
  p.H = Ho; p.W = Wo; p.M = (int64_t)in->n * Ho * Wo;
  p.cout = out->c; p.bias = d->bias; p.post_act = d->post_act;
  p.add = add ? add->data : nullptr; p.add_dtype = add ? add->dtype : GA_F32;
  p.out_bf16 = out_bf16 ? (__nv_bfloat16*)out_bf16->data : nullptr;
  p.out_f32 = out_f32 ? (float*)out_f32->data : nullptr;
  p.mul = d->mul; p.mul_dtype = d->mul_dtype; p.mul_mode = d->mul_mode;
  GA_CHECK(d->dact_out == nullptr || d->dact_dtype == GA_BF16, "ga_conv2d_tc: dact_out must be bf16");
  p.dact = (__nv_bfloat16*)d->dact_out;
  p.act_slope = d->act_slope; p.act_after_add = d->act_after_add;
  p.round_tf32 = (out_f32 && round_tf32_enabled()) ? 1 : 0;
  p.csum = d->csum_out;
  GA_CHECK(d->post_act != GA_ACT_PRELU || d->act_slope != nullptr, "ga_conv2d_tc: PReLU needs act_slope");
  GA_CHECK(d->mul == nullptr || d->mul_mode != GA_MUL_PRELU_FROM_Y || d->act_slope != nullptr, "ga_conv2d_tc: PReLU mask needs act_slope");
  // 3x3 stride-1 convolutions on 64-channel blocks: persistent halo-reuse kernel (conv3x3_tc.cu); -1 = shape not covered there
  if (d->kh == 3 && d->kw == 3 && d->stride == 1 && d->pad == 1 && !in2 && !tf32 && !k32) {
    const int rc = conv3x3_halo_launch(in, d->weight, ktot, out_bf16, out_f32, p, (cudaStream_t)stream);
    if (rc >= 0) return rc;
  }
  // 1x1 stride-1 convolutions / linear layers with a lean epilogue: the same persistent pipeline (resident weights, double-buffered TMEM)
  if (d->kh == 1 && d->kw == 1 && d->stride == 1 && d->pad == 0 && !in2 && !tf32 && !k32 && p.csum == nullptr) {
    const int rc = conv1x1_persistent_launch(in, d->weight, ktot, out_bf16, out_f32, p, (cudaStream_t)stream);
    if (rc >= 0) return rc;
  }
  GA_CHECK(p.csum == nullptr, "ga_conv2d_tc: csum_out requested for a convolution that cannot emit it (ask ga_conv2d_tc_csum_supported first)");
  CUtensorMap tmA, tmA2, tmB;
  if (encode_act_map(&tmA, in, g, d->stride, bk, esize)) return 1;
  if (in2) { if (encode_act_map(&tmA2, in2, g)) return 1; }
  else tmA2 = tmA;
  if (encode_weight_map(&tmB, d->weight, out->c, ktot, block_n, bk, esize)) return 1;

  p.n_blocks = (out->c + block_n - 1) / block_n;
  GA_CHECK(g.m_tiles * p.n_blocks < (int64_t)1 << 31, "ga_conv2d_tc: grid too large");
  dim3 grid((unsigned)(g.m_tiles * p.n_blocks));
  cudaStream_t s = (cudaStream_t)stream;
  // TMA-store epilogue needs 16-byte aligned row pitches and bases; tiny / odd Cout falls back to direct stores
  static int tma_store_enabled = -1;
  if (tma_store_enabled < 0) { const char* e = getenv("GA_TC_TMA_STORE"); tma_store_enabled = e ? atoi(e) : 1; }
  bool tma_ok = tma_store_enabled != 0;
  if (out_bf16 && ((out->c * 2) % 16 != 0 || (((uintptr_t)out_bf16->data) & 15))) tma_ok = false;
  if (out_f32 && ((out->c * 4) % 16 != 0 || (((uintptr_t)out_f32->data) & 15))) tma_ok = false;
  if (block_n == 256 && ((out_bf16 ? 1 : 0) + (out_f32 ? 2 : 0) + (p.dact ? 1 : 0)) > 2) tma_ok = false;   // staging would not fit
  if (p.dact && ((((uintptr_t)p.dact) & 15) || (out->c * 2) % 16 != 0 || (block_n == 32 && out->c > 32))) tma_ok = false;
  if (block_n == 32 && out_bf16 && out->c > 32) tma_ok = false;     // 64-column bf16 panel would spill into the next N tile
  CUtensorMap tmOB = tmA, tmOF = tmA, tmOD = tmA;
  if (tma_ok && p.dact) { if (encode_out_map(&tmOD, p.dact, out->c, p.M, 2)) return 1; }
  if (tma_ok && out_bf16) { if (encode_out_map(&tmOB, out_bf16->data, out->c, p.M, 2)) return 1; }
  if (tma_ok && out_f32) { if (encode_out_map(&tmOF, out_f32->data, out->c, p.M, 4)) return 1; }
  if (g.partial) tma_ok = false;          // a 32-row store box would spill into the next image
  p.tma_store = tma_ok ? 1 : 0;
  p.partial = g.partial;
  const int num_kb = p.taps * p.kc1 + p.kc2;
  static int short_kb = -1;                     // K loops up to this many blocks run on a 2-stage ring -> more co-resident CTAs per SM
  if (short_kb < 0) { const char* e = getenv("GA_TC_SHORT_KB"); short_kb = e ? atoi(e) : 18; }   // measured: 3x3 C=64 @32x32 113 -> 82 us, C=128 @16x16 61 -> 59 us; 36 blocks prefer the deep ring
  const bool short_k = num_kb <= short_kb;
  if (num_kb == 1) {                            // single K block: 1-stage ring, up to 4 CTAs per SM (TMEM-limited)
    switch (block_n) {
      case 32: return launch_tc<32, 1>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
      case 64: return launch_tc<64, 1>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
      case 128: return launch_tc<128, 1>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
      default: break;
    }
  }
  switch (block_n) {
    case 32: return short_k ? launch_tc<32, 2>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s) : launch_tc<32, 4>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
    case 64: return short_k ? launch_tc<64, 2>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s) : launch_tc<64, 4>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
    case 128: return short_k ? launch_tc<128, 2>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s) : launch_tc<128, 3>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
    default: return launch_tc<256, 3>(tmA, tmA2, tmB, tmOB, tmOF, tmOD, p, grid, s);
  }
}

// 1 if ga_conv2d_tc with this descriptor (bf16 output only, no add) can also write the SE channel sums of its output to desc->csum_out
extern "C" int ga_conv2d_tc_csum_supported(const ga_tensor* in, const ga_conv_desc* d, int cout) {
  if (!in || !d || !ga_conv2d_tc_supported(in, nullptr, d, cout)) return 0;
  if (!(d->kh == 3 && d->kw == 3 && d->stride == 1 && d->pad == 1) || d->tf32 || (in->c % 64) != 0) return 0;
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.post_act = d->post_act; p.mul = d->mul; p.dact = (__nv_bfloat16*)d->dact_out; p.act_after_add = d->act_after_add;
  return conv3x3_halo_csum_ok(in, cout, p, true, false) ? 1 : 0;
}
