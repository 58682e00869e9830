// Persistent tcgen05 3x3 convolution with on-chip halo reuse (sm_100a; stride 1, pad 1, bf16 operands, fp32 accumulation in TMEM).
//
// Why a second kernel: conv_tc.cu fetches the activation tile once per filter tap (9 TMA boxes of 16 KB per 128 output pixels and 64 input
// channels) and the weight tile once per CTA.  On B200 the L2 -> SM path delivers ~42 B/clk/SM when all 148 SMs pull (12 TB/s chip-wide),
// and the main-tower convolutions of the NVAE encoder (/root/reference/src/mlvgms_autoencoders/NVAE/modules/architecture.py:96-136) sit
// exactly on that bound: 3x3 C64 @32x32: 216 KB per tile / 42 B/clk = 5.3k clk measured 5.8k, while the MMAs need 1.2k.  This kernel
// cuts the L2 traffic per output pixel 2.5-3x:
//   * the halo tile is loaded ONCE per horizontal tap: 3 boxes of (rows + 2) x W pixels (column-shifted by kx - 1, zero fill = padding)
//     instead of 9; the three vertical taps are three VIEWS of the same box -- a shift by ky image rows is a shift by ky * W * 128 bytes,
//     a multiple of the 1024-byte swizzle atom when W is a multiple of 8, so the UMMA descriptor just starts later;
//   * one CTA owns 256 output pixels (two 128-row accumulators): every weight tile feeds two MMAs;
//   * weights that fit in shared memory (C64 -> 64: 72 KB) are loaded once per CTA and stay resident across all its tiles;
//   * persistent CTAs (one per SM) walk a static tile queue; the TMEM accumulators are double buffered, so the epilogue of tile i
//     (TMEM -> registers -> bias / activation / ... -> swizzled staging -> TMA store) runs under the loads and MMAs of tile i + 1.
// Pipeline stage = (64-channel block, horizontal tap): one halo box (+ the three weight tiles of that column of taps when streaming).
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 = epilogue (shared with conv_tc.cu).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include "ga_common.cuh"
#include "tc_ptx.cuh"
#include "conv_tc_epilogue.cuh"
#include "tc_host.cuh"

namespace ga {

constexpr int C3_THREADS = 192;
constexpr int C3_HDR_BYTES = 1024 + 2048 + 2048 + 4096;   // barriers | bias[<=512] | PReLU slopes[<=512] | channel-sum slabs [2][4][<=128]

struct C3Params {
  int kc;              // 64-channel blocks of Cin
  int W, TR;           // tile width and rows (TR * W == 256): the image width when it is <= 128, 32 x 8 windows of wider images
  int imgW, imgH;      // image size (global pixel indexing)
  int xblocks;         // imgW / W
  int tiles_per_img;   // (H / TR) * xblocks
  int n_mtiles;        // images * tiles_per_img
  int n_tiles;         // n_mtiles * n_blocks
  int stages;          // ring depth
  int a_bytes;         // (TR + 2) * W * 128
  int stage_bytes;     // a_bytes (+ 3 * BLOCK_N * 128 when the weights stream)
  int staging_bytes;   // per epilogue call
  unsigned long long* trace;   // debug (ga_debug_c3_trace): clock64 stamps of CTA 0, [role 3][tile 16][event 16]
};

__device__ __forceinline__ void mbar_arrive1(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// TAPS 9: 3x3 convolution with halo reuse.  TAPS 1: 1x1 convolution / linear layer on the same persistent pipeline -- the activation tensor is a
// plain [M][Cin] matrix, a stage is one 256-row x 64-channel box, tiles may span images (no geometry constraints); what the 1x1 convs gain is
// the persistent structure: resident weights, double-buffered TMEM and the lean epilogues (their tiles are all epilogue).
template <int BLOCK_N, bool RESIDENT_W, int EPI, int TAPS = 9>      // EPI 0: lean epilogue, 1: generic, 2: generic with PReLU / act-after-add, 3: lean + add / mul
__global__ void __launch_bounds__(C3_THREADS, 1) conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                    const __grid_constant__ CUtensorMap tmB,
                                                                    const __grid_constant__ CUtensorMap tmOutB,
                                                                    const __grid_constant__ CUtensorMap tmOutF,
                                                                    const __grid_constant__ CUtensorMap tmOutD, const TcParams p,
                                                                    const C3Params c) {
  constexpr bool GENERAL_ACT = EPI == 2;
  constexpr int B_TILE = BLOCK_N * 128;                       // one tap, one 64-channel block: BLOCK_N rows x 128 B
  constexpr uint32_t TMEM_COLS = 4 * BLOCK_N < 32 ? 32 : 4 * BLOCK_N;   // 2 buffers x 2 sub-tiles
  static_assert(TMEM_COLS <= 512, "TMEM budget");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* hdr = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(hdr);      // [4]
  uint64_t* empty_bar = full_bar + 4;                         // [4]
  uint64_t* tmem_full = empty_bar + 4;                        // [2]
  uint64_t* tmem_empty = tmem_full + 2;                       // [2]
  uint64_t* w_full = tmem_empty + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(w_full + 1);
  float* s_bias = reinterpret_cast<float*>(hdr + 1024);
  float* s_slope = reinterpret_cast<float*>(hdr + 1024 + 2048);
  float* s_csum = reinterpret_cast<float*>(hdr + 1024 + 2048 + 2048);   // double buffered by sub-tile parity
  uint8_t* s_w = hdr + C3_HDR_BYTES;                                           // resident weights: [tap][kc] tiles
  uint8_t* s_ring = s_w + (RESIDENT_W ? TAPS * c.kc * B_TILE : 0);
  uint8_t* s_stage = s_ring + c.stages * c.stage_bytes;                        // epilogue staging (1024-aligned: all sizes are multiples)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_blocks = p.n_blocks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < 4; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
    mbar_init(w_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp >= 2) {
    // bias / slopes of ALL output channels (tiles of different N blocks follow each other in the queue)
    const int et = threadIdx.x - 64;
    for (int i = et; i < n_blocks * BLOCK_N; i += 128) {
      s_bias[i] = (p.bias != nullptr && i < p.cout) ? p.bias[i] : 0.f;
      if (GENERAL_ACT || (EPI == 3 && p.mul_mode == GA_MUL_PRELU_FROM_Y)) s_slope[i] = (p.act_slope != nullptr && i < p.cout) ? p.act_slope[i] : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  auto stamp = [&](int role, int tile_it, int ev) {
    if (c.trace != nullptr && blockIdx.x == 0 && tile_it < 16 && ev < 16)
      c.trace[(role * 16 + tile_it) * 16 + ev] = (unsigned long long)clock64();
  };

  if (warp == 0) {
    // ===================================================================== TMA producer
    if (elect_one_sync()) {
      if (RESIDENT_W) {
        mbar_expect_tx(w_full, TAPS * c.kc * B_TILE);
        for (int tap = 0; tap < TAPS; ++tap)
          for (int kc = 0; kc < c.kc; ++kc)
            tma_load_2d(&tmB, w_full, s_w + (tap * c.kc + kc) * B_TILE, tap * p.cin + kc * 64, 0);
      }
      int stage = 0; uint32_t phase = 0;
      int pit = 0;
      for (int t = blockIdx.x; t < c.n_tiles; t += gridDim.x, ++pit) {
        const int n_blk = t % n_blocks, mt = t / n_blocks;
        if (TAPS == 1) {
          for (int kc = 0; kc < c.kc; ++kc) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            stamp(0, pit, kc);
            mbar_expect_tx(&full_bar[stage], c.stage_bytes);
            uint8_t* dst = s_ring + stage * c.stage_bytes;
            tma_load_2d(&tmA, &full_bar[stage], dst, kc * 64, mt * 256);                    // box = 64 channels x 256 rows (rows past M: zero fill)
            if (!RESIDENT_W) tma_load_2d(&tmB, &full_bar[stage], dst + c.a_bytes, kc * 64, n_blk * BLOCK_N);
            if (++stage == c.stages) { stage = 0; phase ^= 1; }
          }
          continue;
        }
        const int img = mt / c.tiles_per_img, rem = mt - img * c.tiles_per_img;
        const int yb = rem / c.xblocks, y0 = yb * c.TR, x0 = (rem - yb * c.xblocks) * c.W;
        for (int kc = 0; kc < c.kc; ++kc)
          for (int kx = 0; kx < 3; ++kx) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            stamp(0, pit, kc * 3 + kx);
            mbar_expect_tx(&full_bar[stage], c.stage_bytes);
            uint8_t* dst = s_ring + stage * c.stage_bytes;
            tma_load_4d(&tmA, &full_bar[stage], dst, kc * 64, x0 + kx - 1, y0 - 1, img);  // halo box, columns shifted by kx - 1
            if (!RESIDENT_W) {
#pragma unroll
              for (int ky = 0; ky < 3; ++ky)
                tma_load_2d(&tmB, &full_bar[stage], dst + c.a_bytes + ky * B_TILE, (ky * 3 + kx) * p.cin + kc * 64, n_blk * BLOCK_N);
            }
            if (++stage == c.stages) { stage = 0; phase ^= 1; }
          }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    {
      constexpr uint32_t idesc = make_idesc(128, BLOCK_N);
      if (RESIDENT_W) { mbar_wait(w_full, 0); }
      int stage = 0; uint32_t phase = 0;
      uint32_t it = 0;
      // descriptor low words advance by (bytes >> 4): the second sub-tile sits TR/2 image rows further down the halo box, a vertical
      // tap shifts by one image row (W * 128 bytes, a multiple of the 1024-byte swizzle atom)
      const uint32_t sub16 = TAPS == 9 ? ((uint32_t)(c.TR / 2) * c.W * 128) >> 4 : (16384u >> 4);   // 1x1: the second 128 rows of the box
      const uint32_t row16 = TAPS == 9 ? ((uint32_t)c.W * 128) >> 4 : 0u;
      const uint32_t w_lo = smem_desc_lo(smem_u32(s_w));
      for (int t = blockIdx.x; t < c.n_tiles; t += gridDim.x, ++it) {
        const uint32_t buf = it & 1;
        mbar_wait(&tmem_empty[buf], ((it >> 1) & 1) ^ 1);               // epilogue has drained this accumulator pair
        tc_fence_after();
        if (lane == 0) stamp(1, it, 15);
        const uint32_t d0 = tmem_base + buf * (2 * BLOCK_N);
        for (int kc = 0; kc < c.kc; ++kc) {
#pragma unroll 1
          for (int kx = 0; kx < (TAPS == 9 ? 3 : 1); ++kx) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            if (lane == 0) stamp(1, it, kc * 3 + kx);
            const uint32_t a_lo = smem_desc_lo(smem_u32(s_ring + stage * c.stage_bytes));
            const uint32_t b_lo0 = RESIDENT_W ? w_lo + (uint32_t)((kx * c.kc + kc) * (B_TILE >> 4)) : a_lo + (uint32_t)(c.a_bytes >> 4);
            const uint32_t b_step = RESIDENT_W ? (uint32_t)(3 * c.kc * (B_TILE >> 4)) : (uint32_t)(B_TILE >> 4);     // next vertical tap
            const uint32_t acc0 = (kc == 0 && kx == 0) ? 0u : 1u;
            if (elect_one_sync()) {
#pragma unroll
            for (int ky = 0; ky < (TAPS == 9 ? 3 : 1); ++ky) {
              const uint32_t b_lo = b_lo0 + ky * b_step;
#pragma unroll
              for (int s = 0; s < 2; ++s) {
                const uint32_t as_lo = a_lo + s * sub16 + ky * row16;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_bf16(d0 + s * BLOCK_N, smem_desc_from_lo(as_lo + k * 2), smem_desc_from_lo(b_lo + k * 2), idesc,
                            (ky == 0 && k == 0) ? acc0 : 1u);
              }
            }
            umma_commit(&empty_bar[stage]);
            if (kc == c.kc - 1 && kx == (TAPS == 9 ? 2 : 0)) umma_commit(&tmem_full[buf]);
            }
            __syncwarp();
            if (++stage == c.stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
    __syncwarp();
  } else {
    // ===================================================================== epilogue (warps 2..5)
    asm volatile("bar.sync 1, 128;" ::: "memory");   // bias / slopes visible to all epilogue warps
    const int q = warp & 3;
    uint32_t it = 0;
    for (int t = blockIdx.x; t < c.n_tiles; t += gridDim.x, ++it) {
      const int n_blk = t % n_blocks, mt = t / n_blocks;
      const uint32_t buf = it & 1;
      if (warp == 2 && lane == 0) stamp(2, it, 0);
      if (lane == 0) mbar_wait(&tmem_full[buf], (it >> 1) & 1);
      __syncwarp();
      tc_fence_after();
      if (warp == 2 && lane == 0) stamp(2, it, 1);
      // global pixel of the first row of this WARP's 32-row slab, minus q * 32 (the epilogues address pix0 + q * 32 + lane): a slab is 32
      // consecutive pixels of one image row; full-width tiles reduce to mt * 256 + s * 128
      int64_t pixw0 = (int64_t)mt * 256, pixw_s = 128;
      if (TAPS == 9) {
        const int img = mt / c.tiles_per_img, rem = mt - img * c.tiles_per_img;
        const int yb = rem / c.xblocks, y0 = yb * c.TR, x0 = (rem - yb * c.xblocks) * c.W;
        const int rpa = 128 / c.W, r = (q * 32) / c.W, col = (q * 32) - r * c.W;
        pixw0 = ((int64_t)(img * c.imgH + y0 + r) * c.imgW + x0 + col) - q * 32;
        pixw_s = (int64_t)rpa * c.imgW;
      }
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        // this warp's slab of the staging tile is free once its previous bulk stores have read it
        if (lane == 0) tma_store_wait_read();          // this warp's slab of the staging tile is free once its previous bulk stores have read it
        __syncwarp();
        if (warp == 2 && lane == 0) stamp(2, it, 6 + s);
        if (EPI == 0)
          tc_epilogue_lean<BLOCK_N>(p, &tmOutB, &tmOutF, &tmOutD, tmem_base + buf * (2 * BLOCK_N) + s * BLOCK_N, n_blk,
                                    pixw0 + s * pixw_s, s_stage, s_bias + n_blk * BLOCK_N, q, lane, s_csum + s * (4 * BLOCK_N));
        else if (EPI == 3)
          tc_epilogue_lean_am<BLOCK_N>(p, &tmOutB, &tmOutF, tmem_base + buf * (2 * BLOCK_N) + s * BLOCK_N, n_blk,
                                       pixw0 + s * pixw_s, s_stage, s_bias + n_blk * BLOCK_N, s_slope + n_blk * BLOCK_N, q, lane);
        else
          tc_epilogue_tile<BLOCK_N, GENERAL_ACT, true>(p, &tmOutB, &tmOutF, &tmOutD, tmem_base + buf * (2 * BLOCK_N) + s * BLOCK_N, n_blk,
                                                       pixw0 + s * pixw_s, 128, s_stage, s_bias + n_blk * BLOCK_N,
                                                       s_slope + n_blk * BLOCK_N, q, lane);
        if (warp == 2 && lane == 0) stamp(2, it, 2 + s);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive1(&tmem_empty[buf]);
    }
    if (lane == 0) tma_store_wait_all();
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ----------------------------------------------------------------------------- host side
static unsigned long long* g_c3_trace = nullptr;
static int g_halo_enabled = -1;     // GA_TC_HALO / ga_tc_halo_enable: 0 routes every 3x3 conv through the per-tap kernel (A/B comparisons)

template <int BLOCK_N, bool RESIDENT_W, int EPI, int TAPS = 9>
static int launch_c3_(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& ob, const CUtensorMap& of, const CUtensorMap& od,
                      const TcParams& p, const C3Params& c, int smem, int grid, cudaStream_t s) {
  static int configured = 0;
  if (configured < smem) {
    GA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<BLOCK_N, RESIDENT_W, EPI, TAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  conv3x3_tc_kernel<BLOCK_N, RESIDENT_W, EPI, TAPS><<<grid, C3_THREADS, smem, s>>>(a, b, ob, of, od, p, c);
  GA_LAUNCH_OK();
  return 0;
}

template <int BLOCK_N>
static int launch_c3(bool resident, int epi, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& ob, const CUtensorMap& of,
                     const CUtensorMap& od, const TcParams& p, const C3Params& c, int smem, int grid, cudaStream_t s) {
  if (resident) {
    if (epi == 0) return launch_c3_<BLOCK_N, true, 0>(a, b, ob, of, od, p, c, smem, grid, s);
    if (epi == 1) return launch_c3_<BLOCK_N, true, 1>(a, b, ob, of, od, p, c, smem, grid, s);
    if (epi == 3) return launch_c3_<BLOCK_N, true, 3>(a, b, ob, of, od, p, c, smem, grid, s);
    return launch_c3_<BLOCK_N, true, 2>(a, b, ob, of, od, p, c, smem, grid, s);
  }
  if (epi == 0) return launch_c3_<BLOCK_N, false, 0>(a, b, ob, of, od, p, c, smem, grid, s);
  if (epi == 1) return launch_c3_<BLOCK_N, false, 1>(a, b, ob, of, od, p, c, smem, grid, s);
  if (epi == 3) return launch_c3_<BLOCK_N, false, 3>(a, b, ob, of, od, p, c, smem, grid, s);
  return launch_c3_<BLOCK_N, false, 2>(a, b, ob, of, od, p, c, smem, grid, s);
}


// Called by ga_conv2d_tc (conv_tc.cu) with a fully prepared TcParams (epilogue fields, cout, n_blocks unset).
// -> 0 launched, 1 error, -1 not applicable (the caller goes on with the per-tap kernel).
// 1x1 convolutions: lean epilogues only (EPI 0 / 3); anything else stays on the per-tap kernel
template <int BLOCK_N>
static int launch_c1(bool resident, int epi, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& ob, const CUtensorMap& of,
                     const CUtensorMap& od, const TcParams& p, const C3Params& c, int smem, int grid, cudaStream_t s) {
  if (resident) return epi == 0 ? launch_c3_<BLOCK_N, true, 0, 1>(a, b, ob, of, od, p, c, smem, grid, s)
                                : launch_c3_<BLOCK_N, true, 3, 1>(a, b, ob, of, od, p, c, smem, grid, s);
  return epi == 0 ? launch_c3_<BLOCK_N, false, 0, 1>(a, b, ob, of, od, p, c, smem, grid, s)
                  : launch_c3_<BLOCK_N, false, 3, 1>(a, b, ob, of, od, p, c, smem, grid, s);
}

struct C3Plan { C3Params c; int block_n, n_blocks, smem; bool resident; };

// geometry / shared-memory plan of the persistent kernel for one problem; false = shape not covered (the per-tap kernel runs it)
static int wide_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GA_TC_HALO_WIDE"); v = e ? atoi(e) : 1; }
  return v;
}

static bool c3_plan(int n, int H, int W, int cin, int cout, bool out_b, bool out_f, bool dact, bool direct, C3Plan* pl) {
  if (g_halo_enabled < 0) { const char* e = getenv("GA_TC_HALO"); g_halo_enabled = e ? atoi(e) : 1; }
  if (!g_halo_enabled) return false;
  if (cin % 64 != 0 || W % 8 != 0) return false;
  // tile = 256 pixels: TR full rows of an image up to 128 wide, or an 8 x 32 window of a wider one (StyleGAN layers at 256^2 .. 1024^2: the same
  // 40 KB halo boxes and vertical-tap views as a 32 x 32 image, only the box origin and the rows of the output slabs move)
  int TW, TR;
  if (W <= 128 && 256 % W == 0) { TW = W; TR = 256 / W; }
  else if (W % 32 == 0 && wide_enabled()) { TW = 32; TR = 8; }
  else return false;
  if (TR < 2 || TR > H || H % TR != 0) return false;
  if (cout > 512) return false;
  const int block_n = cout <= 32 ? 32 : (cout <= 64 ? 64 : 128);
  const int n_blocks = (cout + block_n - 1) / block_n;
  // TMA-store epilogue only (16-byte aligned row pitches); anything else stays on the per-tap kernel
  if ((out_b || dact) && (cout * 2) % 16 != 0) return false;
  if (out_f && (cout * 4) % 16 != 0) return false;
  C3Params& c = pl->c;
  c.kc = cin / 64; c.W = TW; c.TR = TR; c.imgW = W; c.imgH = H; c.xblocks = W / TW; c.tiles_per_img = (H / TR) * c.xblocks;
  c.n_mtiles = n * c.tiles_per_img;
  c.n_tiles = c.n_mtiles * n_blocks;
  c.a_bytes = (TR + 2) * TW * 128;
  const int b_tile = block_n * 128;
  const int w_bytes = 9 * c.kc * b_tile;
  (void)direct;
  const int staging = ((out_b ? 1 : 0) + (dact ? 1 : 0)) * ((block_n + 63) / 64) * 16384 + (out_f ? (block_n / 32) * 16384 : 0);
  c.staging_bytes = staging;
  const int budget = 227 * 1024 - 1024 - C3_HDR_BYTES - staging;
  // resident weights: one N block, and room for at least 2 ring stages of halo boxes next to them
  const bool resident = n_blocks == 1 && w_bytes + 2 * c.a_bytes <= budget;
  c.stage_bytes = c.a_bytes + (resident ? 0 : 3 * b_tile);
  int stages = (budget - (resident ? w_bytes : 0)) / c.stage_bytes;
  if (stages > 4) stages = 4;
  if (stages < 2) return false;
  c.stages = stages;
  c.trace = g_c3_trace;
  pl->block_n = block_n; pl->n_blocks = n_blocks; pl->resident = resident;
  pl->smem = 1024 + C3_HDR_BYTES + (resident ? w_bytes : 0) + stages * c.stage_bytes + staging;
  return true;
}

static int lean_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GA_TC_LEAN"); v = e ? atoi(e) : 1; }
  return v;
}

// can this 3x3 convolution also emit the SE channel sums of its bf16 output (TcParams::csum)?  Needs the persistent kernel with the lean
// epilogue, no activation / add / mul / tape, bf16 output only, and whole 128-pixel slices per image (the layout of ga_channel_sum)
bool conv3x3_halo_csum_ok(const ga_tensor* in, int cout, const TcParams& p, bool out_b, bool out_f) {
  C3Plan pl;
  if (!lean_enabled() || !out_b || out_f || p.dact || p.add || p.mul || p.post_act != GA_ACT_NONE || p.act_after_add || p.round_tf32) return false;
  if ((in->h * in->w) % 128 != 0) return false;
  return c3_plan(in->n, in->h, in->w, in->c, cout, true, false, false, true, &pl) && pl.c.xblocks == 1;     // (the 128-pixel slices are full-width rows)
}

int conv3x3_halo_launch(const ga_tensor* in, const void* weight, int ktot, const ga_tensor* out_bf16, const ga_tensor* out_f32, TcParams p,
                        cudaStream_t s) {
  const ga_tensor* out = out_bf16 ? out_bf16 : out_f32;
  const int W = in->w, H = in->h, cin = in->c, cout = out->c;
  C3Plan pl;
  p.cin = cin; p.cout = cout; p.tma_store = 1; p.partial = 0;
  const bool general = p.act_after_add != 0 || p.post_act == GA_ACT_PRELU;
  const bool prelu_mask = p.mul != nullptr && p.mul_mode == GA_MUL_PRELU_FROM_Y;     // needs the slopes: lean add/mul epilogue or the general one
  const int epi = general ? 2 : ((lean_enabled() && tc_epilogue_is_lean(p) && !(p.dact && out_f32 && !out_bf16)) ? 0 :
                                 ((lean_enabled() && tc_epilogue_is_lean_am(p)) ? 3 : (prelu_mask ? 2 : 1)));
  if (!c3_plan(in->n, H, W, cin, cout, out_bf16 != nullptr, out_f32 != nullptr, p.dact != nullptr, epi == 0, &pl)) return -1;
  if (out_bf16 && (((uintptr_t)out_bf16->data) & 15)) return -1;
  if (out_f32 && (((uintptr_t)out_f32->data) & 15)) return -1;
  if (p.dact && (((uintptr_t)p.dact) & 15)) return -1;
  const C3Params& c = pl.c;
  const int block_n = pl.block_n, n_blocks = pl.n_blocks, smem = pl.smem, TR = c.TR;
  const bool resident = pl.resident;
  p.cin = cin; p.cout = cout; p.n_blocks = n_blocks; p.M = (int64_t)in->n * H * W; p.H = H; p.W = W;
  p.tma_store = 1; p.partial = 0;

  CUtensorMap tmA, tmB, tmOB, tmOF, tmOD;
  {
    cuuint64_t dims[4] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)in->n};
    cuuint64_t strides[3] = {(cuuint64_t)cin * 2, (cuuint64_t)W * cin * 2, (cuuint64_t)H * W * cin * 2};
    cuuint32_t box[4] = {64u, (cuuint32_t)c.W, (cuuint32_t)(TR + 2), 1u};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if (encode_tiled_cached(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, in->data, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B)) return 1;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)cout};
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t box[2] = {64u, (cuuint32_t)block_n};
    cuuint32_t estr[2] = {1, 1};
    if (encode_tiled_cached(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, weight, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B)) return 1;
  }
  auto out_map = [&](CUtensorMap* tm, void* base, int esize) {
    cuuint64_t dims[2] = {(cuuint64_t)cout, (cuuint64_t)p.M};
    cuuint64_t strides[1] = {(cuuint64_t)cout * esize};
    cuuint32_t box[2] = {(cuuint32_t)(128 / esize), 32u};
    cuuint32_t estr[2] = {1, 1};
    return encode_tiled_cached(tm, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box,
                               estr, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE);
  };
  tmOB = tmA; tmOF = tmA; tmOD = tmA;
  if (out_bf16 && out_map(&tmOB, out_bf16->data, 2)) return 1;
  if (out_f32 && out_map(&tmOF, out_f32->data, 4)) return 1;
  if (p.dact && out_map(&tmOD, p.dact, 2)) return 1;

  if (p.csum != nullptr) GA_CHECK(epi == 0 && conv3x3_halo_csum_ok(in, cout, p, out_bf16 != nullptr, out_f32 != nullptr),
                                  "ga_conv2d_tc: csum_out requested for a convolution that cannot emit it (ask ga_conv2d_tc_csum_supported first)");
  const int grid = c.n_tiles < sm_count() ? c.n_tiles : sm_count();
  switch (block_n) {
    case 32: return launch_c3<32>(resident, epi, tmA, tmB, tmOB, tmOF, tmOD, p, c, smem, grid, s);
    case 64: return launch_c3<64>(resident, epi, tmA, tmB, tmOB, tmOF, tmOD, p, c, smem, grid, s);
    default: return launch_c3<128>(resident, epi, tmA, tmB, tmOB, tmOF, tmOD, p, c, smem, grid, s);
  }
}

// 1x1 / stride 1 convolution (or linear layer) on the persistent pipeline.  -> 0 launched, 1 error, -1 not covered (per-tap kernel runs it).
int conv1x1_persistent_launch(const ga_tensor* in, const void* weight, int ktot, const ga_tensor* out_bf16, const ga_tensor* out_f32, TcParams p,
                              cudaStream_t s) {
  static int enabled = -1;
  if (enabled < 0) { const char* e = getenv("GA_TC_P1X1"); enabled = e ? atoi(e) : 1; }
  if (g_halo_enabled < 0) { const char* e = getenv("GA_TC_HALO"); g_halo_enabled = e ? atoi(e) : 1; }
  if (!enabled || !g_halo_enabled || !lean_enabled()) return -1;
  const ga_tensor* out = out_bf16 ? out_bf16 : out_f32;
  const int cin = in->c, cout = out->c;
  const int64_t M = (int64_t)in->n * in->h * in->w;
  if (cin % 64 != 0 || ktot != cin || cout > 512 || M < 256 * 64) return -1;      // small problems: launch-bound either way, keep the per-tap kernel
  if ((out_bf16 || p.dact) && (cout * 2) % 16 != 0) return -1;
  if (out_f32 && (cout * 4) % 16 != 0) return -1;
  if (out_bf16 && (((uintptr_t)out_bf16->data) & 15)) return -1;
  if (out_f32 && (((uintptr_t)out_f32->data) & 15)) return -1;
  if (p.dact && (((uintptr_t)p.dact) & 15)) return -1;
  p.cin = cin; p.cout = cout; p.tma_store = 1; p.partial = 0; p.M = M; p.H = in->h; p.W = in->w;
  if (p.act_after_add != 0 || p.post_act == GA_ACT_PRELU || (p.mul != nullptr && p.mul_mode == GA_MUL_PRELU_FROM_Y)) return -1;
  int epi;
  if (tc_epilogue_is_lean(p) && !(p.dact && out_f32 && !out_bf16)) epi = 0;
  // add/mul epilogues stream one more tensor per output row: with one CTA per SM and four epilogue warps too few of those loads are in flight
  // (N=384 dgrad*mul at 32x32: 425 us here against 273 us on the per-tap kernel, which keeps several CTAs per SM) -- GA_TC_P1X1=2 opts them in.
  else if (enabled >= 2 && tc_epilogue_is_lean_am(p)) epi = 3;
  else return -1;
  const int block_n = cout <= 32 ? 32 : (cout <= 64 ? 64 : 128);
  const int n_blocks = (cout + block_n - 1) / block_n;
  p.n_blocks = n_blocks;
  C3Params c;
  memset(&c, 0, sizeof(c));
  c.kc = cin / 64; c.W = 0; c.TR = 0; c.tiles_per_img = 1; c.imgW = 0; c.imgH = 0; c.xblocks = 1;
  c.n_mtiles = (int)((M + 255) / 256);
  c.n_tiles = c.n_mtiles * n_blocks;
  c.a_bytes = 256 * 128;
  const int b_tile = block_n * 128;
  const int w_bytes = c.kc * b_tile;
  const int staging = ((out_bf16 ? 1 : 0) + (p.dact ? 1 : 0)) * ((block_n + 63) / 64) * 16384 + (out_f32 ? (block_n / 32) * 16384 : 0);
  c.staging_bytes = staging;
  const int budget = 227 * 1024 - 1024 - C3_HDR_BYTES - staging;
  const bool resident = n_blocks == 1 && w_bytes + 2 * c.a_bytes <= budget;
  c.stage_bytes = c.a_bytes + (resident ? 0 : b_tile);
  int stages = (budget - (resident ? w_bytes : 0)) / c.stage_bytes;
  if (stages > 4) stages = 4;
  if (stages < 2) return -1;
  c.stages = stages;
  c.trace = nullptr;
  const int smem = 1024 + C3_HDR_BYTES + (resident ? w_bytes : 0) + stages * c.stage_bytes + staging;
  CUtensorMap tmA, tmB, tmOB, tmOF, tmOD;
  {
    cuuint64_t dims[2] = {(cuuint64_t)cin, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)cin * 2};
    cuuint32_t box[2] = {64u, 256u};
    cuuint32_t estr[2] = {1, 1};
    if (encode_tiled_cached(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, in->data, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B)) return 1;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)cout};
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t box[2] = {64u, (cuuint32_t)block_n};
    cuuint32_t estr[2] = {1, 1};
    if (encode_tiled_cached(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, weight, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B)) return 1;
  }
  auto out_map = [&](CUtensorMap* tm, void* base, int esize) {
    cuuint64_t dims[2] = {(cuuint64_t)cout, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)cout * esize};
    cuuint32_t box[2] = {(cuuint32_t)(128 / esize), 32u};
    cuuint32_t estr[2] = {1, 1};
    return encode_tiled_cached(tm, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box,
                               estr, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE);
  };
  tmOB = tmA; tmOF = tmA; tmOD = tmA;
  if (out_bf16 && out_map(&tmOB, out_bf16->data, 2)) return 1;
  if (out_f32 && out_map(&tmOF, out_f32->data, 4)) return 1;
  if (p.dact && out_map(&tmOD, p.dact, 2)) return 1;
  const int grid = c.n_tiles < sm_count() ? c.n_tiles : sm_count();
  switch (block_n) {
    case 32: return launch_c1<32>(resident, epi, tmA, tmB, tmOB, tmOF, tmOD, p, c, smem, grid, s);
    case 64: return launch_c1<64>(resident, epi, tmA, tmB, tmOB, tmOF, tmOD, p, c, smem, grid, s);
    default: return launch_c1<128>(resident, epi, tmA, tmB, tmOB, tmOF, tmOD, p, c, smem, grid, s);
  }
}

}  // namespace ga

// debug: clock64 timeline of CTA 0 of the halo kernel (scripts/trace_conv3x3.py); buf = device uint64[3 * 16 * 16] or NULL (off)
extern "C" int ga_debug_c3_trace(unsigned long long* buf) {
  ga::g_c3_trace = buf;
  return 0;
}

// debug / A-B testing: 1 = persistent halo kernel for the shapes it covers (default), 0 = per-tap kernel everywhere
extern "C" int ga_tc_halo_enable(int on) {
  ga::g_halo_enabled = on ? 1 : 0;
  return 0;
}
