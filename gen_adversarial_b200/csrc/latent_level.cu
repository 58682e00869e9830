// Tail of one NVAE decoder latent level in ONE tcgen05 kernel (NVAE/model.py:226-256): prior sampler -> latent mix -> decoder combiner.
//
//   pp  = dec_sampler(ELU(x))                    GEMM 1: A = x_elu (bf16 ELU copy written by the last cell's se_residual), N = 2 * zdim
//   z   = mix(muq, pp, eps, alpha)               epilogue warps, one pixel row per thread, from TMEM; z goes to shared memory only
//   out = dec_comb([xa | z])                     GEMM 2: K blocks of xa by TMA, then the z tile; fp32 stream + bf16 copy by TMA store
//
// Per 128-pixel tile this reads x_elu, xa and muq once and writes the new stream once; `pp` (fp32, 2 * zdim channels) and `z` no longer make
// a round trip through HBM (pp is written only when a taping forward asks for it).  Results are bit-identical to the three-launch path:
//   * GEMM 1 runs N = 64 MMAs over the same 64-channel K blocks as the 1x1 kernels (block_n 64 for the 40 sampler channels), + bias in fp32;
//   * the latent mix is the same device function as latent_mix (ga_common.cuh: latent_mix_prior, latent_eps4);
//   * GEMM 2 runs the per-tap kernel's MMA shapes (N = min(C, 128) per instruction) in its K order: the xa blocks, then z.  The per-tap
//     kernel multiplies z as a 64-channel block whose upper 32 channels are zero; here z is a 32-channel block (64-byte swizzle), which skips
//     two MMAs that add exact zeros.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 = latent mix and output epilogue.
// TMEM: at C = 64, pp has its own 64 columns and GEMM 2's xa blocks run while the epilogue warps mix z; at C = 128 / 256 GEMM 2 re-uses GEMM 1's
// columns (pp has been read before z exists).  3 CTAs per SM at C <= 128 (2 at C = 256), so one CTA's serial chain overlaps the others'.  fp32 mode, level 0 and the encoder-side convolutions stay on their own kernels.
#include <cuda.h>
#include "ga_common.cuh"
#include "tc_ptx.cuh"
#include "tc_host.cuh"

namespace ga {

constexpr int LL_THREADS = 192;
constexpr int LL_A_BYTES = 128 * 64 * 2;            // one 64-channel K block of 128 pixels (128-byte swizzle)
constexpr int LL_SAMPLER_N = 64;                    // MMA width of GEMM 1 (2 * zdim <= 64 sampler channels, zero rows above)
constexpr int LL_ZMAX = 32;                         // z channels in the z K block (zdim <= 32; zero above zdim)
constexpr int LL_Z_BYTES = 128 * LL_ZMAX * 2;       // 8 KB, 64-byte swizzle
constexpr int LL_GROUP_BYTES = 16384 + 32768;       // output staging of 64 columns: one bf16 panel + two fp32 panels
constexpr int LL_HDR = 2048;                        // barriers, TMEM address, both biases

template <int C>
struct LLCfg {
  // pp lives in its own TMEM columns where the allocation stays small enough for 3 CTAs per SM (C = 64: 128 columns), so GEMM 2's xa blocks
  // run while the epilogue warps mix z; at C = 128 / 256 GEMM 2 re-uses GEMM 1's columns and waits for the mix
  static constexpr int PP_COL = C == 64 ? 64 : 0;
  static constexpr int KC = C / 64;                 // 64-channel K blocks of x_elu (GEMM 1) and of xa (GEMM 2)
  static constexpr int BN2 = C < 128 ? C : 128;     // N per GEMM-2 MMA (the per-tap kernel's block_n)
  static constexpr int STAGES = 2;
  static constexpr int STAGE_BYTES = LL_A_BYTES + C * 128;   // A block + the widest B block (C rows of GEMM 2)
  static constexpr int RING = STAGES * STAGE_BYTES;
  // output staging re-uses the ring once GEMM 2 has retired: 1 buffer (C = 64, 128) or 2 (C = 256, the stores of one 64-column group
  // drain while the next is written)
  static constexpr int NBUF = (RING / LL_GROUP_BYTES) < KC ? (RING / LL_GROUP_BYTES) : KC;
  static constexpr uint32_t TMEM_COLS = C == 64 ? 128 : C;
  static constexpr int SMEM = 1024 + LL_HDR + RING + LL_Z_BYTES;
};

struct LLParams {
  int64_t M;                   // pixels
  int HW;                      // pixels per image
  int zdim;                    // latent channels; GEMM 1 has 2 * zdim = [mu_p | logsig_p]
  int cq;                      // channels (row pitch) of muq
  const float* muq;            // [M][cq] fp32, first zdim channels used
  const float* eps;            // NCHW [n][zdim][HW] fp32, or nullptr = Philox
  float* pp;                   // [M][2 * zdim] fp32 (taping), or nullptr
  const float* b1;             // sampler bias [2 * zdim]
  const float* b2;             // combiner bias [C]
  const float* alpha;          // device scalar
  float temp;
  SeedArg seed;
  int level;
  int64_t sample0;
};

// ZG: zdim / 4 (a template parameter so that the per-pixel latent arrays hold exactly zdim values).  3 CTAs per SM at C <= 128 and zdim <= 20
// (96 registers, no spills); 2 otherwise (more registers than 3 CTAs leave would spill)
template <int C, int ZG>
__global__ void __launch_bounds__(LL_THREADS, (C == 256 || ZG > 5) ? 2 : 3) latent_level_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmXa,
                                                                     const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                                                                     const __grid_constant__ CUtensorMap tmW2z, const __grid_constant__ CUtensorMap tmOB,
                                                                     const __grid_constant__ CUtensorMap tmOF, const LLParams p) {
  using K = LLCfg<C>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* hdr = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = hdr + LL_HDR;
  uint8_t* ztile = ring + K::RING;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(hdr);
  uint64_t* empty_bar = full_bar + K::STAGES;
  uint64_t* pp_full = empty_bar + K::STAGES;        // GEMM 1 retired
  uint64_t* z_ready = pp_full + 1;                  // the 4 epilogue warps have read pp and written z
  uint64_t* acc_full = z_ready + 1;                 // GEMM 2 retired
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(acc_full + 1);
  float* s_b1 = reinterpret_cast<float*>(hdr + 128);            // 64 floats
  float* s_b2 = reinterpret_cast<float*>(hdr + 128 + 256);      // C floats
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int pix0 = (int)blockIdx.x * 128;
  constexpr int NUM_KB = 2 * K::KC + 1;             // GEMM 1 blocks, GEMM 2 xa blocks, GEMM 2 z-weight block

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX); tma_prefetch_desc(&tmXa); tma_prefetch_desc(&tmW1); tma_prefetch_desc(&tmW2); tma_prefetch_desc(&tmW2z);
    for (int i = 0; i < K::STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(pp_full, 1);
    mbar_init(z_ready, 4);
    mbar_init(acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(K::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================================================================== TMA producer
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < NUM_KB; ++kb) {
      if (elect_one_sync()) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* a_dst = ring + stage * K::STAGE_BYTES;
        uint8_t* b_dst = a_dst + LL_A_BYTES;
        if (kb < K::KC) {
          mbar_expect_tx(&full_bar[stage], LL_A_BYTES + LL_SAMPLER_N * 128);
          tma_load_2d(&tmX, &full_bar[stage], a_dst, kb * 64, pix0);
          tma_load_2d(&tmW1, &full_bar[stage], b_dst, kb * 64, 0);
        } else if (kb < 2 * K::KC) {
          mbar_expect_tx(&full_bar[stage], LL_A_BYTES + C * 128);
          tma_load_2d(&tmXa, &full_bar[stage], a_dst, (kb - K::KC) * 64, pix0);
          tma_load_2d(&tmW2, &full_bar[stage], b_dst, (kb - K::KC) * 64, 0);
        } else {
          mbar_expect_tx(&full_bar[stage], C * LL_ZMAX * 2);
          tma_load_2d(&tmW2z, &full_bar[stage], b_dst, C, 0);       // combiner weight columns C .. C + 31 (zero beyond zc)
        }
      }
      __syncwarp();
      if (++stage == K::STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    constexpr uint32_t idesc1 = make_idesc(128, LL_SAMPLER_N);
    constexpr uint32_t idesc2 = make_idesc(128, K::BN2);
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < NUM_KB; ++kb) {
      if (elect_one_sync()) {
        // z must be in shared memory before its block; with shared TMEM columns, pp must also have been read before GEMM 2 starts
        if (kb == (K::PP_COL != 0 ? NUM_KB - 1 : K::KC)) { mbar_wait(z_ready, 0); tc_fence_after(); }
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(ring + stage * K::STAGE_BYTES);
        const uint32_t b_addr = a_addr + LL_A_BYTES;
        if (kb < K::KC) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_base + K::PP_COL, smem_desc_from_lo(smem_desc_lo(a_addr) + k * 2), smem_desc_from_lo(smem_desc_lo(b_addr) + k * 2), idesc1,
                      (kb > 0 || k > 0) ? 1u : 0u);
        } else if (kb < 2 * K::KC) {
#pragma unroll
          for (int nc = 0; nc < C / K::BN2; ++nc)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_base + nc * K::BN2, smem_desc_from_lo(smem_desc_lo(a_addr) + k * 2),
                        smem_desc_from_lo(smem_desc_lo(b_addr + nc * K::BN2 * 128) + k * 2), idesc2, (kb > K::KC || k > 0) ? 1u : 0u);
        } else {
          const uint32_t z_addr = smem_u32(ztile);
#pragma unroll
          for (int nc = 0; nc < C / K::BN2; ++nc)
#pragma unroll
            for (int k = 0; k < 2; ++k)
              umma_bf16(tmem_base + nc * K::BN2, make_smem_desc_sw64(z_addr + k * 32), make_smem_desc_sw64(b_addr + nc * K::BN2 * 64 + k * 32),
                        idesc2, 1u);
        }
        umma_commit(&empty_bar[stage]);
        if (kb == K::KC - 1) umma_commit(pp_full);
        if (kb == NUM_KB - 1) umma_commit(acc_full);
      }
      __syncwarp();
      if (++stage == K::STAGES) { stage = 0; phase ^= 1; }
    }
  } else {
    // ===================================================================== latent mix + output epilogue (warps 2..5)
    const int et = threadIdx.x - 64;
    if (et < LL_SAMPLER_N) s_b1[et] = et < 2 * p.zdim ? p.b1[et] : 0.f;
    for (int i = et; i < C; i += 128) s_b2[i] = p.b2[i];
    asm volatile("bar.sync 1, 128;" ::: "memory");
    const int q = warp & 3;                          // TMEM lane quadrant of this warp
    const int row = q * 32 + lane;
    const int64_t pix = (int64_t)pix0 + row;
    const bool row_ok = pix < p.M;
    const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
    constexpr int Z = 4 * ZG;

    // muq and eps while GEMM 1 runs
    float mq[Z], ee[Z];
    {
      const int64_t n = pix / p.HW;
      const int hw = (int)(pix - n * p.HW);
      const uint64_t seed = p.seed.get();
#pragma unroll
      for (int j = 0; j < ZG; ++j) {
        float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
        float e4[4] = {0.f, 0.f, 0.f, 0.f};
        if (row_ok) {
          m4 = __ldg(reinterpret_cast<const float4*>(p.muq + pix * p.cq + 4 * j));
          if (p.eps != nullptr) {
#pragma unroll
            for (int u = 0; u < 4; ++u) e4[u] = __ldg(p.eps + (n * Z + 4 * j + u) * p.HW + hw);
          } else {
            latent_eps4(seed, noise_stream(p.sample0 + n, p.level + 1), j, hw, p.HW, e4);
          }
        }
        mq[4 * j] = m4.x; mq[4 * j + 1] = m4.y; mq[4 * j + 2] = m4.z; mq[4 * j + 3] = m4.w;
#pragma unroll
        for (int u = 0; u < 4; ++u) ee[4 * j + u] = e4[u];
      }
    }
    const float a = *p.alpha;

    if (lane == 0) mbar_wait(pp_full, 0);
    __syncwarp();
    tc_fence_after();
    // mu_p of group j sits in columns 4j.., logsig_p in Z + 4j..: runtime TMEM addresses, compile-time registers
    uint32_t rp[ZG][4], rl[ZG][4];
#pragma unroll
    for (int j = 0; j < ZG; ++j) { tmem_ld4(t_row + K::PP_COL + 4 * j, rp[j]); tmem_ld4(t_row + K::PP_COL + Z + 4 * j, rl[j]); }
    tmem_ld_wait();
    uint32_t zp[LL_ZMAX / 2];                        // z as bf16 pairs, zero above zdim (K padding of GEMM 2)
#pragma unroll
    for (int j = 0; j < LL_ZMAX / 4; ++j) {
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      if (j < ZG) {
        float mp[4], lp[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          mp[u] = __uint_as_float(rp[j][u]) + s_b1[4 * j + u];
          lp[u] = __uint_as_float(rl[j][u]) + s_b1[Z + 4 * j + u];
          o[u] = latent_mix_prior(a, mq[4 * j + u], mp[u], lp[u], ee[4 * j + u], p.temp);
        }
        if (p.pp != nullptr && row_ok) {
          float* pr = p.pp + pix * (2 * Z);
          *reinterpret_cast<float4*>(pr + 4 * j) = make_float4(mp[0], mp[1], mp[2], mp[3]);
          *reinterpret_cast<float4*>(pr + Z + 4 * j) = make_float4(lp[0], lp[1], lp[2], lp[3]);
        }
      }
      zp[2 * j] = pack_bf16x2(o[0], o[1]);
      zp[2 * j + 1] = pack_bf16x2(o[2], o[3]);
    }
    {
      // K-major, 64-byte swizzle (what TMA writes for a 32-channel SWIZZLE_64B box): 16-byte chunk c of row r at r * 64 + ((c ^ ((r >> 1) & 3)) << 4)
      uint8_t* zrow = ztile + row * 64;
      const uint32_t sw = (uint32_t)((row >> 1) & 3);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        *reinterpret_cast<uint4*>(zrow + ((c ^ sw) << 4)) = make_uint4(zp[4 * c], zp[4 * c + 1], zp[4 * c + 2], zp[4 * c + 3]);
    }
    fence_proxy_async_smem();                        // z visible to the tensor core (async proxy)
    tc_fence_before();                               // pp reads ordered before GEMM 2 overwrites the columns
    __syncwarp();
    if (lane == 0) mbar_arrive(z_ready);

    if (lane == 0) mbar_wait(acc_full, 0);
    __syncwarp();
    tc_fence_after();
    // output: 64 columns at a time, staged in the idle ring (SWIZZLE_128B box layout of the store maps), each warp stores its 32-row slab
    const uint32_t sw = (uint32_t)(row & 7);
#pragma unroll 1
    for (int g = 0; g < K::KC; ++g) {
      uint8_t* buf = ring + (g % K::NBUF) * LL_GROUP_BYTES;
      if (g >= K::NBUF) {                            // this warp's slab of `buf` must have been read by its earlier stores
        if (lane == 0) tma_store_wait_read_n<K::NBUF - 1>();
        __syncwarp();
      }
      uint32_t rr[4][16];
#pragma unroll
      for (int i = 0; i < 4; ++i) tmem_ld16(t_row + g * 64 + i * 16, rr[i]);
      tmem_ld_wait();
#pragma unroll
      for (int ci = 0; ci < 4; ++ci) {
        const int c0 = g * 64 + ci * 16;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[ci][j]) + s_b2[c0 + j];
        uint8_t* pb = buf + row * 128;
        const uint32_t kb0 = (uint32_t)(ci * 2);
        *reinterpret_cast<uint4*>(pb + ((kb0 ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        *reinterpret_cast<uint4*>(pb + (((kb0 + 1) ^ sw) << 4)) =
            make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
        uint8_t* pf = buf + 16384 + (ci >> 1) * 16384 + row * 128;
        const uint32_t kf0 = (uint32_t)((ci & 1) * 4);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(pf + (((kf0 + j) ^ sw) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {                               // TMA clips rows >= M (partial last tile)
        const int row0 = pix0 + q * 32;
        tma_store_2d(&tmOB, buf + q * 32 * 128, g * 64, row0);
        tma_store_2d(&tmOF, buf + 16384 + q * 32 * 128, g * 64, row0);
        tma_store_2d(&tmOF, buf + 32768 + q * 32 * 128, g * 64 + 32, row0);
        tma_store_commit();
      }
      __syncwarp();
    }
    if (lane == 0) tma_store_wait_read();            // shared memory stays valid until the bulk stores have read it
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(K::TMEM_COLS) : "memory");
  }
}

static int ll_encode_2d(CUtensorMap* tm, CUtensorMapDataType dt, int esize, const void* base, int inner, int64_t rows, int box_inner, int box_rows,
                        CUtensorMapSwizzle sw, CUtensorMapL2promotion l2) {
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)inner * esize};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return encode_tiled_cached(tm, dt, 2, base, dims, strides, box, estr, sw, l2);
}

template <int C, int ZG>
static int launch_latent_level(const ga_tensor* x_elu, const ga_tensor* xa, const void* w_sampler, const void* w_comb, int zc,
                               const ga_tensor* out_bf16, const ga_tensor* out_f32, const LLParams& p, cudaStream_t s) {
  using K = LLCfg<C>;
  constexpr auto BF = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUtensorMap tmX, tmXa, tmW1, tmW2, tmW2z, tmOB, tmOF;
  if (ll_encode_2d(&tmX, BF, 2, x_elu->data, C, p.M, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B)) return 1;
  if (ll_encode_2d(&tmXa, BF, 2, xa->data, C, p.M, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B)) return 1;
  if (ll_encode_2d(&tmW1, BF, 2, w_sampler, C, 2 * p.zdim, 64, LL_SAMPLER_N, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B)) return 1;
  if (ll_encode_2d(&tmW2, BF, 2, w_comb, C + zc, C, 64, C, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B)) return 1;
  if (ll_encode_2d(&tmW2z, BF, 2, w_comb, C + zc, C, LL_ZMAX, C, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B)) return 1;
  if (ll_encode_2d(&tmOB, BF, 2, out_bf16->data, C, p.M, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE)) return 1;
  if (ll_encode_2d(&tmOF, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out_f32->data, C, p.M, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_NONE)) return 1;
  static bool configured = false;
  if (!configured) {
    GA_CUDA(cudaFuncSetAttribute(latent_level_kernel<C, ZG>, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM));
    configured = true;
  }
  latent_level_kernel<C, ZG><<<(unsigned)((p.M + 127) / 128), LL_THREADS, K::SMEM, s>>>(tmX, tmXa, tmW1, tmW2, tmW2z, tmOB, tmOF, p);
  GA_LAUNCH_OK();
  return 0;
}

// (C, zdim / 4) -> instantiation; ZG runs 1 .. LL_ZMAX / 4
template <int ZG>
static int dispatch_c(int C, int zg, const ga_tensor* x_elu, const ga_tensor* xa, const void* w_sampler, const void* w_comb, int zc,
                      const ga_tensor* out_bf16, const ga_tensor* out_f32, const LLParams& p, cudaStream_t s) {
  if constexpr (ZG < LL_ZMAX / 4) {
    if (zg != ZG) return dispatch_c<ZG + 1>(C, zg, x_elu, xa, w_sampler, w_comb, zc, out_bf16, out_f32, p, s);
  }
  switch (C) {
    case 64: return launch_latent_level<64, ZG>(x_elu, xa, w_sampler, w_comb, zc, out_bf16, out_f32, p, s);
    case 128: return launch_latent_level<128, ZG>(x_elu, xa, w_sampler, w_comb, zc, out_bf16, out_f32, p, s);
    default: return launch_latent_level<256, ZG>(x_elu, xa, w_sampler, w_comb, zc, out_bf16, out_f32, p, s);
  }
}

}  // namespace ga

using namespace ga;

static bool ll_aligned(const void* ptr) { return (((uintptr_t)ptr) & 15) == 0; }

extern "C" int ga_latent_level(const ga_tensor* x_elu, const ga_tensor* xa, const ga_tensor* muq, const float* eps_nchw, const void* w_sampler,
                               const float* b_sampler, const void* w_comb, const float* b_comb, int zc, uint64_t seed, int level, int64_t sample0,
                               const float* alpha_dev, float temperature, int zdim, const ga_tensor* out_bf16, const ga_tensor* out_f32,
                               const ga_tensor* pp_out, void* stream) {
  GA_CHECK(x_elu && xa && muq && w_sampler && b_sampler && w_comb && b_comb && alpha_dev && out_bf16 && out_f32, "ga_latent_level: null argument");
  const int C = xa->c;
  GA_CHECK(C == 64 || C == 128 || C == 256, "ga_latent_level: %d channels (64, 128 or 256 supported)", C);
  GA_CHECK(x_elu->dtype == GA_BF16 && xa->dtype == GA_BF16 && same_shape(x_elu, xa), "ga_latent_level: x_elu and xa must be bf16 of one shape");
  GA_CHECK(out_bf16->dtype == GA_BF16 && out_f32->dtype == GA_F32 && same_shape(out_bf16, xa) && same_shape(out_f32, xa),
           "ga_latent_level: outputs must be bf16 / fp32 of the input's shape");
  GA_CHECK(zdim >= 4 && zdim <= LL_ZMAX && zdim % 4 == 0, "ga_latent_level: zdim %d (a multiple of 4 up to %d)", zdim, LL_ZMAX);
  GA_CHECK(zc >= zdim && zc <= LL_ZMAX && zc % 8 == 0, "ga_latent_level: combiner z channels %d", zc);
  GA_CHECK(muq->dtype == GA_F32 && muq->n == xa->n && muq->h == xa->h && muq->w == xa->w && muq->c >= zdim && muq->c % 4 == 0,
           "ga_latent_level: muq must be fp32 [n][h][w][>= zdim, multiple of 4]");
  GA_CHECK(!pp_out || (pp_out->dtype == GA_F32 && pp_out->n == xa->n && pp_out->h == xa->h && pp_out->w == xa->w && pp_out->c == 2 * zdim),
           "ga_latent_level: pp_out must be fp32 [n][h][w][2 * zdim]");
  GA_CHECK(ll_aligned(x_elu->data) && ll_aligned(xa->data) && ll_aligned(muq->data) && ll_aligned(w_sampler) && ll_aligned(w_comb) &&
               ll_aligned(out_bf16->data) && ll_aligned(out_f32->data) && (!pp_out || ll_aligned(pp_out->data)),
           "ga_latent_level: tensors must be 16-byte aligned");
  LLParams p;
  p.M = (int64_t)xa->n * xa->h * xa->w;
  if (p.M == 0) return 0;
  GA_CHECK(p.M < ((int64_t)1 << 31) - 128, "ga_latent_level: too many pixels");
  p.HW = xa->h * xa->w; p.zdim = zdim; p.cq = muq->c;
  p.muq = (const float*)muq->data; p.eps = eps_nchw; p.pp = pp_out ? (float*)pp_out->data : nullptr;
  p.b1 = b_sampler; p.b2 = b_comb; p.alpha = alpha_dev; p.temp = temperature;
  cudaStream_t s = (cudaStream_t)stream;
  p.seed = make_seed(seed, s); p.level = level; p.sample0 = sample0;
  return dispatch_c<1>(C, zdim / 4, x_elu, xa, w_sampler, w_comb, zc, out_bf16, out_f32, p, s);
}
