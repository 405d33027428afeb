// K4 on the tensor cores — nn.Upsample(scale_factor=2, mode='trilinear', align_corners=True) (med3d.py:83, 86)
// of an NDHWC 16-bit tensor as a small GEMM per output brick:
//
//     out[128 voxels x C] = Wt[128 voxels x 96 source voxels] . in_patch[96 source voxels x C]
//
// The CUDA-core kernel (aux_kernels.cu) needs ~100 instructions per 16 bytes of output for the fp32
// interpolation arithmetic and is issue-bound at ~2.3 TB/s; the interpolation itself is linear, so here
//   * an output brick of 8 x 4 x 4 voxels reads a source patch of at most 6 x 4 x 4 voxels (one TMA box per
//     64-channel chunk, SWIZZLE_128B rows of 64 channels = the MN-major B operand of tcgen05.mma);
//   * four warps generate the brick's interpolation matrix Wt (eight non-zeros per row: the products of ATen's
//     three per-axis weights, computed in fp32 and rounded once to the storage type) straight into the K-major
//     SWIZZLE_128B A-operand layout; it is reused for every channel chunk of the brick;
//   * six M128 x N64 x K16 MMAs per chunk accumulate in TMEM; the epilogue rounds to the storage type, stages
//     the 128 x 64 tile in shared memory and sends it with one TMA store.
// The kernel moves 16 KiB of output per ~450 tensor-core clocks per SM: HBM-bound.
// Rounding: the reference rounds nothing (fp32); K4 rounds the result once to the storage type; this kernel
// additionally rounds the eight weights to the storage type (relative 2^-12 each for fp16, 2^-9 for bf16).
//
// Roles (320 threads): warps 0-3 epilogue, warp 4 lane 0 TMA producer, warp 5 MMA issuer (owns TMEM),
// warps 6-9 interpolation-matrix generators.
#include "umma_common.cuh"

namespace dram {

static constexpr int U_TW = 8, U_TH = 4, U_TD = 4;             // output brick (w, h, d) = 128 voxels
static constexpr int U_PW = 6, U_PH = 4, U_PD = 4;             // source patch = 96 voxels = K
static constexpr int U_K = U_PW * U_PH * U_PD;                 // 96
static constexpr int U_B_BYTES = U_K * 128;                    // 12 KiB per 64-channel chunk
static constexpr int U_B_STAGES = 6;
static constexpr int U_W_BYTES = 2 * 128 * 128;                // two 64-wide K atoms x 128 rows = 32 KiB
static constexpr int U_OUT_BYTES = 128 * 128;                  // 16 KiB staged output tile
static constexpr int U_ACC = 4;                                // TMEM accumulators of 64 columns
static constexpr int U_THREADS = 320;
static constexpr int U_PRODUCER_WARP = 4, U_MMA_WARP = 5, U_GEN_WARP0 = 6;
static constexpr int U_SMEM_BYTES = 1024 + U_B_STAGES * U_B_BYTES + 2 * U_W_BYTES + 2 * U_OUT_BYTES + 256;

struct UpParams {
  int n, Dl, Hl, Wl, D, H, W, C;     // low-resolution and output dims, channels
  int chunks;                        // C / 64
  int tiles_w, tiles_h, tiles_d, tiles_per_sample, total_tiles;
  float sd, sh, sw;                  // ATen source scales
  int is_f16;                        // storage type of in / out (the interpolation matrix is always fp16)
  const int *items, *count;          // optional work list: tiles items[0 .. *count) instead of all (null = all)
};

struct UpTile {
  int sample, w0, h0, d0;            // output brick origin
  int wl0, hl0, dl0;                 // source patch origin
};
__device__ __forceinline__ UpTile decode_up_tile(const UpParams &p, int tile) {
  UpTile t;
  t.sample = tile / p.tiles_per_sample;
  int r = tile - t.sample * p.tiles_per_sample;
  const int iw = r % p.tiles_w;
  r /= p.tiles_w;
  const int ih = r % p.tiles_h;
  const int id = r / p.tiles_h;
  t.w0 = iw * U_TW; t.h0 = ih * U_TH; t.d0 = id * U_TD;
  t.wl0 = lin_index_ac(t.w0, p.sw, p.Wl).i0;
  t.hl0 = lin_index_ac(t.h0, p.sh, p.Hl).i0;
  t.dl0 = lin_index_ac(t.d0, p.sd, p.Dl).i0;
  return t;
}

// kind::f16 instruction descriptor with an MN-major B operand (bit 16); A and B must have the same 16-bit type
// (mixing an fp16 A with a bf16 B is an illegal instruction), so the interpolation matrix uses the storage type.
__host__ __device__ constexpr uint32_t make_idesc_up(int n, int is_f16) {
  return (1u << 4) | ((is_f16 ? 0u : 1u) << 7) | ((is_f16 ? 0u : 1u) << 10) | (1u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(128 >> 4) << 24);
}

__global__ void __launch_bounds__(U_THREADS, 1)
upsample2x_umma_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_out,
                       const __grid_constant__ UpParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = smem_base + U_B_STAGES * U_B_BYTES;
  const uint32_t out_base = w_base + 2 * U_W_BYTES;
  const uint32_t bar_base = out_base + 2 * U_OUT_BYTES;
  auto b_addr = [&](int s) { return smem_base + (uint32_t)s * U_B_BYTES; };
  auto w_addr = [&](int s) { return w_base + (uint32_t)s * U_W_BYTES; };
  auto out_addr = [&](int s) { return out_base + (uint32_t)s * U_OUT_BYTES; };
  auto b_full = [&](int s) { return bar_base + 8u * s; };
  auto b_empty = [&](int s) { return bar_base + 8u * (U_B_STAGES + s); };
  auto w_full = [&](int s) { return bar_base + 8u * (2 * U_B_STAGES + s); };
  auto w_empty = [&](int s) { return bar_base + 8u * (2 * U_B_STAGES + 2 + s); };
  auto t_full = [&](int a) { return bar_base + 8u * (2 * U_B_STAGES + 4 + a); };
  auto t_empty = [&](int a) { return bar_base + 8u * (2 * U_B_STAGES + 4 + U_ACC + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * U_B_STAGES + 4 + 2 * U_ACC);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < U_B_STAGES; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(b_empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(w_full(s), 128);
      mbar_init(w_empty(s), 1);
    }
    for (int a = 0; a < U_ACC; ++a) {
      mbar_init(t_full(a), 1);
      mbar_init(t_empty(a), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == U_MMA_WARP) tmem_alloc(tmem_slot, U_ACC * 64);
  if (warp == U_PRODUCER_WARP && lane == 0) prefetch_tensormap(&map_in);
  if (threadIdx.x == 0) prefetch_tensormap(&map_out);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
  // CTA b runs positions b, b + grid, ... of the work list (of all tiles without one)
  const int total = p.items ? *p.count : p.total_tiles;
  auto tile_at = [&](int i) { return p.items ? __ldg(p.items + i) : i; };

  if (warp == U_PRODUCER_WARP) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int i = blockIdx.x; i < total; i += gridDim.x) {
        const UpTile t = decode_up_tile(p, tile_at(i));
        for (int c = 0; c < p.chunks; ++c) {
          mbar_wait(b_empty(stage), phase ^ 1u);
          mbar_expect_tx(b_full(stage), U_B_BYTES);
          tma_load_5d(b_addr(stage), &map_in, b_full(stage), c * 64, t.wl0, t.hl0, t.dl0, t.sample);
          if (++stage == U_B_STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == U_MMA_WARP) {
    const uint32_t idesc = make_idesc_up(64, p.is_f16);
    int stage = 0, acc = 0, wi = 0;
    uint32_t phase = 0, acc_phase = 0, w_phase = 0;
    for (int i = blockIdx.x; i < total; i += gridDim.x) {
      mbar_wait(w_full(wi), w_phase);
      tcgen05_fence_after();
      for (int c = 0; c < p.chunks; ++c) {
        mbar_wait(t_empty(acc), acc_phase ^ 1u);
        mbar_wait(b_full(stage), phase);
        tcgen05_fence_after();
        if (elect_one_sync()) {
#pragma unroll
          for (int j = 0; j < U_K / 16; ++j) {
            // A: interpolation matrix, K-major, atom j / 4, 32 bytes per K step inside the 128-byte row
            const uint64_t da = make_sw128_desc(w_addr(wi) + (uint32_t)((j >> 2) * (128 * 128) + (j & 3) * 32));
            // B: source patch, MN-major: 16 source voxels = 16 rows of 128 bytes per K step
            const uint64_t db = make_sw128_desc(b_addr(stage) + (uint32_t)(j * 16 * 128));
            umma_bf16(tmem_base + (uint32_t)(acc * 64), da, db, idesc, j > 0 ? 1u : 0u);
          }
          umma_commit(b_empty(stage));
          umma_commit(t_full(acc));
          if (c == p.chunks - 1) umma_commit(w_empty(wi));
        }
        __syncwarp();
        if (++stage == U_B_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
        if (++acc == U_ACC) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
      if (++wi == 2) {
        wi = 0;
        w_phase ^= 1u;
      }
    }
  } else if (warp >= U_GEN_WARP0) {
    // ------------------------------- interpolation-matrix generators -------------------------------
    const int r = threadIdx.x - U_GEN_WARP0 * 32;  // output voxel (row) of the brick
    const int lw = r & (U_TW - 1), lh = (r >> 3) & (U_TH - 1), ld = r >> 5;
    // Both matrices start as zeros (cooperative, conflict-free); afterwards a thread only clears the (at most)
    // eight entries its row had in the brick that used the buffer before.
    for (int i = r; i < 2 * U_W_BYTES / 16; i += 128)
      asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(w_base + 16u * i), "r"(0u) : "memory");
    asm volatile("bar.sync 2, 128;" ::: "memory");
    uint32_t prev0[8], prev1[8];  // per buffer: addresses of this row's entries in the brick before
#pragma unroll
    for (int q = 0; q < 8; ++q) prev0[q] = prev1[q] = 0xffffffffu;
    auto generate = [&](const UpTile &t, uint32_t wbuf, uint32_t (&mine)[8]) {
      const uint32_t base = wbuf + (uint32_t)r * 128u;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (mine[q] != 0xffffffffu) asm volatile("st.shared.u16 [%0], %1;" ::"r"(mine[q]), "h"((unsigned short)0) : "memory");
        mine[q] = 0xffffffffu;
      }
      const int od = t.d0 + ld, oh = t.h0 + lh, ow = t.w0 + lw;
      if (od < p.D && oh < p.H && ow < p.W) {
        LinIdx ix[3] = {lin_index_ac(od, p.sd, p.Dl), lin_index_ac(oh, p.sh, p.Hl), lin_index_ac(ow, p.sw, p.Wl)};
#pragma unroll
        for (int a = 0; a < 3; ++a)
          if (ix[a].i1 == ix[a].i0) {  // clamped at the last source voxel: both weights belong to it
            ix[a].w0 += ix[a].w1;
            ix[a].w1 = 0.0f;
          }
#pragma unroll
        for (int cd = 0; cd < 2; ++cd)
#pragma unroll
          for (int chh = 0; chh < 2; ++chh)
#pragma unroll
            for (int cw = 0; cw < 2; ++cw) {
              const float wt = (cd ? ix[0].w1 : ix[0].w0) * ((chh ? ix[1].w1 : ix[1].w0) * (cw ? ix[2].w1 : ix[2].w0));
              if ((cd && ix[0].i1 == ix[0].i0) || (chh && ix[1].i1 == ix[1].i0) || (cw && ix[2].i1 == ix[2].i0)) continue;
              const int zd = (cd ? ix[0].i1 : ix[0].i0) - t.dl0, zh = (chh ? ix[1].i1 : ix[1].i0) - t.hl0;
              const int zw = (cw ? ix[2].i1 : ix[2].i0) - t.wl0;
              const int k = (zd * U_PH + zh) * U_PW + zw;  // row of the patch box: w fastest, then h, then d
              const int kk = k & 63;
              const uint32_t addr = base + (uint32_t)((k >> 6) * 128 * 128) + (uint32_t)((((kk >> 3) ^ (r & 7)) << 4) + (kk & 7) * 2);
              unsigned short bits;
              if (p.is_f16) {
                const __half hv = __float2half_rn(wt);
                bits = *reinterpret_cast<const unsigned short *>(&hv);
              } else {
                const __nv_bfloat16 hv = __float2bfloat16_rn(wt);
                bits = *reinterpret_cast<const unsigned short *>(&hv);
              }
              asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(bits) : "memory");
              mine[cd * 4 + chh * 2 + cw] = addr;
            }
      }
    };
    int wi = 0;
    uint32_t w_phase = 0;
    for (int i = blockIdx.x; i < total; i += gridDim.x) {
      const UpTile t = decode_up_tile(p, tile_at(i));
      mbar_wait(w_empty(wi), w_phase ^ 1u);
      if (wi == 0) generate(t, w_addr(0), prev0);
      else generate(t, w_addr(1), prev1);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(w_full(wi));
      if (++wi == 2) {
        wi = 0;
        w_phase ^= 1u;
      }
    }
  } else {
    // ------------------------------- epilogue warps 0..3 -------------------------------
    const int row = warp * 32 + lane;
    int acc = 0, gi = 0;
    uint32_t acc_phase = 0;
    for (int i = blockIdx.x; i < total; i += gridDim.x) {
      const UpTile t = decode_up_tile(p, tile_at(i));
      for (int c = 0; c < p.chunks; ++c, ++gi) {
        const int b = gi & 1;
        mbar_wait(t_full(acc), acc_phase);
        tcgen05_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t)(acc * 64) + ((uint32_t)(warp * 32) << 16);
        uint32_t v0[32], v1[32];
        tmem_ld_32x32b_x32(taddr, v0);
        tmem_ld_32x32b_x32(taddr + 32u, v1);
        if (threadIdx.x == 0) tma_store_wait_read<1>();  // the store that last read out tile b is done with it
        asm volatile("bar.sync 1, 128;" ::: "memory");
        tmem_wait_ld();
        tcgen05_fence_before();
        mbar_arrive(t_empty(acc));  // the accumulator is in registers: hand it back
        const uint32_t orow = out_addr(b) + (uint32_t)row * 128u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t *v = j < 4 ? v0 : v1;
          const int o = (j & 3) * 8;
          const uint32_t chunk = (uint32_t)((j ^ (row & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(orow + chunk),
                       "r"(pack2(__uint_as_float(v[o + 0]), __uint_as_float(v[o + 1]), p.is_f16)),
                       "r"(pack2(__uint_as_float(v[o + 2]), __uint_as_float(v[o + 3]), p.is_f16)),
                       "r"(pack2(__uint_as_float(v[o + 4]), __uint_as_float(v[o + 5]), p.is_f16)),
                       "r"(pack2(__uint_as_float(v[o + 6]), __uint_as_float(v[o + 7]), p.is_f16))
                       : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (threadIdx.x == 0) {
          tma_store_5d(&map_out, out_addr(b), c * 64, t.w0, t.h0, t.d0, t.sample);
          tma_store_commit();
        }
        if (++acc == U_ACC) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == U_MMA_WARP) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, U_ACC * 64);
  }
}

}  // namespace dram

using namespace dram;

struct dram_upsample_plan {
  CUtensorMap map_in, map_out;
  UpParams p;
};

// Largest source extent under any aligned window of `win` outputs (same fp32 index arithmetic as the device).
static int up_max_span(int out_size, int in_size, int win) {
  const float scale = ac_scale(in_size, out_size);
  int worst = 0;
  for (int o0 = 0; o0 < out_size; o0 += win) {
    const int o1 = o0 + win - 1 > out_size - 1 ? out_size - 1 : o0 + win - 1;
    int lo = (int)(scale * (float)o0);
    if (lo > in_size - 1) lo = in_size - 1;
    int hi = (int)(scale * (float)o1);
    if (hi > in_size - 1) hi = in_size - 1;
    if (hi < in_size - 1) hi += 1;
    if (hi - lo + 1 > worst) worst = hi - lo + 1;
  }
  return worst;
}

extern "C" int dram_upsample2x_plan_create(const void *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                                           int32_t c, int32_t dtype, dram_upsample_plan **plan) {
  DRAM_REQUIRE(plan, "dram_upsample2x_plan_create: null plan pointer");
  *plan = nullptr;
  DRAM_REQUIRE(x && out, "dram_upsample2x_plan_create: null pointer");
  DRAM_REQUIRE(n > 0 && d > 0 && h > 0 && w > 0 && c > 0 && c % 64 == 0,
               "dram_upsample2x_plan_create: bad shape (c must be a multiple of 64)");
  DRAM_REQUIRE(dtype == DRAM_DTYPE_BF16 || dtype == DRAM_DTYPE_F16, "dram_upsample2x_plan_create: bad dtype");
  const int D = 2 * d, H = 2 * h, W = 2 * w;
  DRAM_REQUIRE(up_max_span(D, d, U_TD) <= U_PD && up_max_span(H, h, U_TH) <= U_PH && up_max_span(W, w, U_TW) <= U_PW,
               "dram_upsample2x_plan_create: source patch exceeds %dx%dx%d", U_PD, U_PH, U_PW);
  dram_upsample_plan *pl = new dram_upsample_plan();
  memset(pl, 0, sizeof(*pl));
  UpParams &p = pl->p;
  p.n = n; p.Dl = d; p.Hl = h; p.Wl = w; p.D = D; p.H = H; p.W = W; p.C = c;
  p.chunks = c / 64;
  p.tiles_w = ceil_div(W, U_TW); p.tiles_h = ceil_div(H, U_TH); p.tiles_d = ceil_div(D, U_TD);
  p.tiles_per_sample = p.tiles_w * p.tiles_h * p.tiles_d;
  const int64_t total = (int64_t)p.tiles_per_sample * n;
  if (total > 0x7fffffffLL) {
    delete pl;
    set_error("dram_upsample2x_plan_create: too many tiles");
    return DRAM_E_ARG;
  }
  p.total_tiles = (int)total;
  p.sd = ac_scale(d, D); p.sh = ac_scale(h, H); p.sw = ac_scale(w, W);
  p.is_f16 = dtype == DRAM_DTYPE_F16;
  int rc = encode_act_map(&pl->map_in, x, n, d, h, w, c, 64, U_PW, U_PH, U_PD, 1, 1, 1, p.is_f16);
  if (rc == DRAM_OK) rc = encode_act_map(&pl->map_out, out, n, D, H, W, c, 64, U_TW, U_TH, U_TD, 1, 1, 1, p.is_f16);
  if (rc == DRAM_OK)
    rc = check_cuda(cudaFuncSetAttribute(upsample2x_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         U_SMEM_BYTES),
                    "cudaFuncSetAttribute(upsample2x_umma_kernel)");
  if (rc != DRAM_OK) {
    delete pl;
    return rc;
  }
  *plan = pl;
  return DRAM_OK;
}

extern "C" int dram_upsample2x_plan_destroy(dram_upsample_plan *plan) {
  delete plan;
  return DRAM_OK;
}

static int upsample_launch(const dram_upsample_plan *plan, const int *items, const int *count, int32_t max_ctas,
                           void *stream) {
  int ctas = sm_count();
  if (max_ctas > 0 && max_ctas < ctas) ctas = max_ctas;
  if (plan->p.total_tiles < ctas) ctas = plan->p.total_tiles;
  UpParams p = plan->p;
  p.items = items;
  p.count = count;
  upsample2x_umma_kernel<<<ctas, U_THREADS, U_SMEM_BYTES, reinterpret_cast<cudaStream_t>(stream)>>>(
      plan->map_in, plan->map_out, p);
  DRAM_CHECK_LAUNCH("upsample2x_umma_kernel launch");
  return DRAM_OK;
}

extern "C" int dram_upsample2x_plan_run(const dram_upsample_plan *plan, int32_t max_ctas, void *stream) {
  DRAM_REQUIRE(plan, "dram_upsample2x_plan_run: null plan");
  return upsample_launch(plan, nullptr, nullptr, max_ctas, stream);
}

extern "C" int dram_upsample2x_worklist_size(const dram_upsample_plan *plan, int32_t *entries) {
  DRAM_REQUIRE(plan && entries, "dram_upsample2x_worklist_size: null argument");
  *entries = plan->p.total_tiles;
  return DRAM_OK;
}

// Work items: the 8 x 4 x 4 output bricks, numbered with W fastest.
extern "C" int dram_upsample2x_worklist(const dram_upsample_plan *plan, const uint32_t *support, int32_t radius,
                                        uint8_t *flags, int32_t *tiles, int32_t *count, void *stream) {
  DRAM_REQUIRE(plan, "dram_upsample2x_worklist: null plan");
  const UpParams &p = plan->p;
  return worklist_build(support, p.n, p.D, p.H, p.W, U_TW, U_TH, U_TD, 0, radius, flags, tiles, count, p.total_tiles,
                        reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int dram_upsample2x_plan_run_listed(const dram_upsample_plan *plan, const int32_t *tiles,
                                               const int32_t *count, int32_t max_ctas, void *stream) {
  DRAM_REQUIRE(plan && tiles && count, "dram_upsample2x_plan_run_listed: null argument");
  return upsample_launch(plan, tiles, count, max_ctas, stream);
}
