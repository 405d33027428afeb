// K1 — conv3d as an implicit GEMM on the sm_100a tensor cores.
//
//   A (activations) : NDHWC bf16.  One TMA box load per (filter tap, 64-channel chunk)
//                     fetches the tap-shifted [td][th][tw][64] brick of the input straight
//                     into the canonical K-major SWIZZLE_128B UMMA layout (128 rows x 128 B).
//                     Zero padding = TMA out-of-bounds fill; dilation = tap offset;
//                     stride = tensor-map elementStrides.  A second tensor map supplies the
//                     channels of the skip tensor, so cat([up(x), skip]) is never built
//                     (med3d.py:39-48, 85-89).
//   B (weights)     : bf16 [Cout][tap][Cin] (K-major), BatchNorm scale folded in, one 2-D TMA
//                     box per K-chunk.
//   D (accumulator) : fp32 in TMEM, two buffers of BLOCK_N columns so the epilogue of tile i
//                     overlaps the MMAs of tile i+1.
//   Epilogue        : tcgen05.ld -> +bias -> +residual (full, or shortcut type A: strided
//                     read, channels < res_c only; med3d.py:103-112,141) -> ReLU -> bf16
//                     NDHWC store; for the 32-channel us3 layer optionally the 1x1x1 heads
//                     (+sigmoid) in fp32 (med3d.py:329-332, 382 / 230-233, 283).
//
// Roles (192 threads): warps 0-3 epilogue (TMEM lane quarter = warp id), warp 4 lane 0 TMA
// producer, warp 5 lane 0 MMA issuer (warp 5 also owns the TMEM allocation).
// Persistent: grid <= #SMs, tile = blockIdx.x + i * gridDim.x, n-tile fastest.
// Filter taps whose whole brick lies in the zero padding are skipped by producer and issuer.
#include "umma_common.cuh"
#include "conv_plan.h"

namespace dram {

static constexpr int BLOCK_M = 128;       // output voxels per tile == TMEM lanes
static constexpr int BLOCK_K = 64;        // bf16 channels per K-chunk == one 128-byte swizzle row
static constexpr int UMMA_K = 16;         // K per tcgen05.mma for 16-bit inputs
static constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KiB
static constexpr int NUM_THREADS = 192;
static constexpr int NUM_THREADS_STAGED = 320;               // + warps 6-9: second half of the epilogue columns
static constexpr int PRODUCER_WARP = 4;
static constexpr int MMA_WARP = 5;

static constexpr int EPI_TILE_BYTES = BLOCK_M * 128;         // staged epilogue: 128 rows x 64 channels
static constexpr int RES_BUFS = 4;                           // residual tiles in flight (DRAM latency ~ 3 groups)

// STAGED: the epilogue goes through shared memory and TMA (coalesced stores, residual tiles loaded by TMA)
// instead of one 16-byte global access per lane and row.  Used for the 1x1x1 convolutions of the bottleneck
// blocks, which are bound by exactly those accesses (K is at most 32 chunks), with BLOCK_N <= 128 so that four
// operand stages, two output tiles and four residual tiles fit in shared memory together.
// BLOCK_N = 256 staged: for 1x1x1 convolutions WITHOUT a residual (K13's low-resolution product, the bottleneck blocks'
// first convolution): no residual tiles, three operand stages of 48 KiB.
template <int BLOCK_N, bool STAGED = false>
struct ConvCfg {
  static constexpr int B_STAGE_BYTES = BLOCK_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int STAGES = STAGED ? (BLOCK_N == 256 ? 3 : 4) : ((BLOCK_N <= 64) ? 8 : (BLOCK_N == 128 ? 6 : 4));
  static constexpr int TMEM_COLS = (2 * BLOCK_N < 32) ? 32 : 2 * BLOCK_N;
  static constexpr int RES_TILES = BLOCK_N == 256 ? 0 : RES_BUFS;
  static constexpr int EPI_BYTES = STAGED ? (2 + RES_TILES) * EPI_TILE_BYTES : 0;  // output + residual tiles
  // 1 KiB alignment slack + stages + epilogue tiles + barriers
  static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + EPI_BYTES + 256;
};

template <int BLOCK_N, bool STAGED>
__global__ void __launch_bounds__(STAGED ? NUM_THREADS_STAGED : NUM_THREADS, 1)
conv3d_umma_kernel(const __grid_constant__ CUtensorMap map_a1,
                   const __grid_constant__ CUtensorMap map_a2,
                   const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_out,
                   const __grid_constant__ CUtensorMap map_res, const __grid_constant__ ConvKParams p) {
  using Cfg = ConvCfg<BLOCK_N, STAGED>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B operands need 1 KiB alignment.
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t epi_base = smem_base + STAGES * Cfg::STAGE_BYTES;  // STAGED: out[2], res[2] tiles of 16 KiB
  const uint32_t bar_base = epi_base + Cfg::EPI_BYTES;
  auto out_tile = [&](int b) { return epi_base + (uint32_t)b * EPI_TILE_BYTES; };
  auto res_tile = [&](int b) { return epi_base + (uint32_t)(2 + b) * EPI_TILE_BYTES; };
  auto res_full = [&](int q, int b) { return bar_base + 8u * (2 * STAGES + 5 + q * RES_BUFS + b); };  // q < 4, b < RES_BUFS
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tmem_full_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tmem_empty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  auto smem_a = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };
  auto smem_b = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + A_STAGE_BYTES; };

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full_bar(a), 1);
      mbar_init(tmem_empty_bar(a), STAGED ? 256 : 128);
    }
    if (STAGED)
      for (int b = 0; b < 4 * RES_BUFS; ++b) mbar_init(res_full(0, b), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  if (warp == PRODUCER_WARP && lane == 0) {
    prefetch_tensormap(&map_a1);
    prefetch_tensormap(&map_a2);
    prefetch_tensormap(&map_w);
  }
  if (STAGED && threadIdx.x == 0) {
    prefetch_tensormap(&map_out);
    prefetch_tensormap(&map_res);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);  // provably warp-uniform

  if (warp == PRODUCER_WARP) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile, BLOCK_N);
        for (int zd = 0; zd < p.kd; ++zd) {
          const int id0 = t.d0 * p.sd + zd * p.dd - p.pd;
          if (tap_is_padding(id0, p.td, p.sd, p.Di)) continue;
          for (int zh = 0; zh < p.kh; ++zh) {
            const int ih0 = t.h0 * p.sh + zh * p.dh - p.ph;
            if (tap_is_padding(ih0, p.th, p.sh, p.Hi)) continue;
            for (int zw = 0; zw < p.kw; ++zw) {
              const int iw0 = t.w0 * p.sw + zw * p.dw - p.pw;
              if (tap_is_padding(iw0, p.tw, p.sw, p.Wi)) continue;
              const int tap = (zd * p.kh + zh) * p.kw + zw;
              for (int ch = 0; ch < p.chunks_total; ++ch) {
                mbar_wait(empty_bar(stage), phase ^ 1u);
                mbar_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
                if (ch < p.chunks1)
                  tma_load_5d(smem_a(stage), &map_a1, full_bar(stage), ch * BLOCK_K, iw0, ih0, id0,
                              t.sample);
                else
                  tma_load_5d(smem_a(stage), &map_a2, full_bar(stage), (ch - p.chunks1) * BLOCK_K,
                              iw0, ih0, id0, t.sample);
                tma_load_2d(smem_b(stage), &map_w, full_bar(stage),
                            (tap * p.chunks_total + ch) * BLOCK_K, t.n0);
                if (++stage == STAGES) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == MMA_WARP) {
    {  // the whole warp walks the loops (uniform control flow); one elected lane issues
      const uint32_t idesc = make_idesc_16bit(BLOCK_M, BLOCK_N, p.epi.is_f16);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile, BLOCK_N);
        mbar_wait(tmem_empty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        uint32_t accumulate = 0;
        for (int zd = 0; zd < p.kd; ++zd) {
          if (tap_is_padding(t.d0 * p.sd + zd * p.dd - p.pd, p.td, p.sd, p.Di)) continue;
          for (int zh = 0; zh < p.kh; ++zh) {
            if (tap_is_padding(t.h0 * p.sh + zh * p.dh - p.ph, p.th, p.sh, p.Hi)) continue;
            for (int zw = 0; zw < p.kw; ++zw) {
              if (tap_is_padding(t.w0 * p.sw + zw * p.dw - p.pw, p.tw, p.sw, p.Wi)) continue;
              for (int ch = 0; ch < p.chunks_total; ++ch) {
                mbar_wait(full_bar(stage), phase);
                tcgen05_fence_after();
                const uint64_t da = make_sw128_desc(smem_a(stage));
                const uint64_t db = make_sw128_desc(smem_b(stage));
                if (elect_one_sync()) {
#pragma unroll
                  for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                    // +32 bytes along K inside the 128-byte swizzle row = +2 in the >>4 address field
                    umma_bf16(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc,
                              (k > 0) ? 1u : accumulate);
                  }
                  umma_commit(empty_bar(stage));  // frees the smem stage when these MMAs retire
                }
                __syncwarp();
                accumulate = 1;
                if (++stage == STAGES) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
            }
          }
        }
        if (elect_one_sync()) umma_commit(tmem_full_bar(acc));  // accumulator complete -> epilogue
        __syncwarp();
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
    __syncwarp();
  } else if (STAGED) {
    // ------------------------------- epilogue warps 0..3 and 6..9, staged through shared memory + TMA -------------
    // Work unit = one 64-channel group of one tile ("group", gi counts them across this CTA's tiles).
    // Eight warps: warp w works on TMEM lane quarter w % 4 (rows 32*(w%4) ...), warps 0-3 on the first 32 columns of
    // the group, warps 6-9 on the second 32.  The two warps of a quarter own that quarter's 32 rows of the tiles: one
    // of their lanes keeps RES_BUFS residual slices (4 KiB each) in flight and sends the finished output slice with its
    // own TMA store (tensor-map box = the 32 voxels of the quarter), and the pair meets at a 64-thread named barrier.
    // Round 2, ncu of 64 -> 256 + residual at 100x128x128 (profiles/conv_1x1_r2k1.md): with ONE thread storing whole
    // tiles and two 256-thread barriers per group the epilogue warps showed a quarter of their samples at those
    // barriers.  Measured after this change: 0.475 -> 0.472 ms (4.0 TB/s of compulsory bytes) — the waits were a
    // symptom, the layer is bound by its 0.84 GB write + 1.05 GB read stream; kept because it needs no CTA-wide barrier.
    constexpr int GROUPS = BLOCK_N >= 64 ? BLOCK_N / 64 : 1;
    constexpr uint32_t SLICE_BYTES = EPI_TILE_BYTES / 4;
    const int quarter = warp & 3, half = warp < 4 ? 0 : 1;
    const int row = quarter * 32 + lane;
    const bool storer = half == 0 && lane == 0;
    // where the quarter's first row sits inside the tw x th x td brick
    const int row0 = quarter * 32;
    const int qw = row0 & (p.tw - 1), qh = (row0 >> p.tw_log2) & (p.th - 1), qd = row0 >> (p.tw_log2 + p.th_log2);
    const bool has_res = p.staged_res != 0;
    const int my_tiles = p.total_tiles > (int)blockIdx.x ? (p.total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int total_groups = my_tiles * GROUPS;
    auto pair_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory"); };
    auto issue_res = [&](int gi) {  // the quarter's storer only
      if (!has_res || gi >= total_groups) return;
      const int tile = blockIdx.x + (gi / GROUPS) * gridDim.x;
      const TileCoord t = decode_tile(p, tile, BLOCK_N);
      const int rb = gi % RES_BUFS;
      mbar_expect_tx(res_full(quarter, rb), SLICE_BYTES);
      const int rs = p.epi.res_stride;
      tma_load_5d(res_tile(rb) + (uint32_t)quarter * SLICE_BYTES, &map_res, res_full(quarter, rb),
                  t.n0 + (gi % GROUPS) * 64, (t.w0 + qw) * rs, (t.h0 + qh) * rs, (t.d0 + qd) * rs, t.sample);
    };
    if (storer)
      for (int g0 = 0; g0 < RES_BUFS; ++g0) issue_res(g0);
    int acc = 0, gi = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile, BLOCK_N);
      mbar_wait(tmem_full_bar(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)(acc * BLOCK_N) + ((uint32_t)(quarter * 32) << 16);
#pragma unroll 1
      for (int g = 0; g < GROUPS; ++g, ++gi) {
        const int b = gi & 1, rb = gi % RES_BUFS;
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + (uint32_t)(g * 64 + half * 32), v);
        if (has_res) mbar_wait(res_full(quarter, rb), (uint32_t)((gi / RES_BUFS) & 1));
        // the store that last read this quarter of out_tile(b) (group gi - 2) must be done with shared memory
        if (storer) tma_store_wait_read<1>();
        pair_sync();
        tmem_wait_ld();
        epilogue_group_staged(p.epi, v, t.n0 + g * 64 + half * 32, row, half, res_tile(rb), has_res, out_tile(b));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        pair_sync();
        if (storer) {
          if (t.w0 + qw < p.Wo && t.h0 + qh < p.Ho && t.d0 + qd < p.Do)  // a quarter of a border tile can lie outside
            tma_store_5d(&map_out, out_tile(b) + (uint32_t)quarter * SLICE_BYTES, t.n0 + g * 64, t.w0 + qw, t.h0 + qh,
                         t.d0 + qd, t.sample);
          tma_store_commit();  // one bulk group per group even when nothing is stored (wait_group.read 1 counts them)
          issue_res(gi + RES_BUFS);  // both warps of the quarter have read its slice of res_tile(rb)
        }
      }
      tcgen05_fence_before();
      mbar_arrive(tmem_empty_bar(acc));
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1u;
      }
    }
    if (storer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before exit
  } else {
    // ------------------------------- epilogue warps 0..3 -------------------------------
    const int row = warp * 32 + lane;  // TMEM lane == row of the 128-voxel tile
    const int lw = row & (p.tw - 1);
    const int lh = (row >> p.tw_log2) & (p.th - 1);
    const int ld = row >> (p.tw_log2 + p.th_log2);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile, BLOCK_N);
      const int od = t.d0 + ld, oh = t.h0 + lh, ow = t.w0 + lw;
      const bool valid = (od < p.Do) && (oh < p.Ho) && (ow < p.Wo);
      const uint16_t *res_row = residual_row(p.epi, valid, t.sample, od, oh, ow);
      ResGroup res = load_residual_group(p.epi, res_row, t.n0);  // in flight while this warp waits for the accumulator
      mbar_wait(tmem_full_bar(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)(acc * BLOCK_N) + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + (uint32_t)c0, v);
        const ResGroup next = load_residual_group(p.epi, c0 + 32 < BLOCK_N ? res_row : nullptr, t.n0 + c0 + 32);
        tmem_wait_ld();
        if (valid) epilogue_group<BLOCK_N == 32>(p.epi, v, t.n0 + c0, t.sample, od, oh, ow, res);
        res = next;
      }
      tcgen05_fence_before();
      mbar_arrive(tmem_empty_bar(acc));  // 128 arrivals hand the accumulator back to the issuer
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1u;
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------
// Host side: tensor maps + plan
// ----------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void *sym = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || sym == nullptr) {
    cudaGetLastError();
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

// NDHWC activation tensor as a 5-D map (C, W, H, D, N); box = box_c channels x bw x bh x bd voxels.
int encode_act_map(CUtensorMap *map, const void *base, int n, int d, int h, int w, int c, int box_c, int bw,
                   int bh, int bd, int sw, int sh, int sd, int is_f16) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available (no CUDA driver?)");
    return DRAM_E_DRIVER;
  }
  cuuint64_t gdim[5] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)d, (cuuint64_t)n};
  cuuint64_t gstr[4] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2,
                        (cuuint64_t)d * h * w * c * 2};
  // With a traversal stride s the box spans (t-1)*s+1 input elements and lands t of them.
  cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)((bw - 1) * sw + 1),
                       (cuuint32_t)((bh - 1) * sh + 1), (cuuint32_t)((bd - 1) * sd + 1), 1};
  cuuint32_t estr[5] = {1, (cuuint32_t)sw, (cuuint32_t)sh, (cuuint32_t)sd, 1};
  CUresult r = enc(map, is_f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5,
                   const_cast<void *>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(activation %dx%dx%dx%dx%d box %dx%dx%d stride %d,%d,%d) -> %d",
              n, d, h, w, c, bw, bh, bd, sw, sh, sd, (int)r);
    return DRAM_E_DRIVER;
  }
  return DRAM_OK;
}

// NDHWC activation tensor, un-swizzled rows of box_c channels: box = box_c x bw x bh voxels of one plane.
int encode_act_map_plain(CUtensorMap *map, const void *base, int n, int d, int h, int w, int c, int box_c, int bw,
                         int bh, int is_f16) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available (no CUDA driver?)");
    return DRAM_E_DRIVER;
  }
  cuuint64_t gdim[5] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)d, (cuuint64_t)n};
  cuuint64_t gstr[4] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2,
                        (cuuint64_t)d * h * w * c * 2};
  cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)bw, (cuuint32_t)bh, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(map, is_f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5,
                   const_cast<void *>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(plain activation %dx%dx%dx%dx%d box %dx%d) -> %d", n, d, h, w, c, bw, bh, (int)r);
    return DRAM_E_DRIVER;
  }
  return DRAM_OK;
}

int encode_weight_map(CUtensorMap *map, const void *base, int cout, int64_t ktot, int block_n, int is_f16) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available (no CUDA driver?)");
    return DRAM_E_DRIVER;
  }
  cuuint64_t gdim[2] = {(cuuint64_t)ktot, (cuuint64_t)cout};
  cuuint64_t gstr[1] = {(cuuint64_t)ktot * 2};
  cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)block_n};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, is_f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                   const_cast<void *>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(weight %d x %lld, box_n %d) -> %d", cout, (long long)ktot,
              block_n, (int)r);
    return DRAM_E_DRIVER;
  }
  return DRAM_OK;
}

static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}
static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

static int conv_out(int in, int k, int s, int d, int p) { return (in + 2 * p - d * (k - 1) - 1) / s + 1; }

// M256 tile kernel (conv3d_pair.cu)
int pair_plan_wanted(const dram_conv_desc *d, int block_n, int64_t k_chunks, int64_t m_tiles, int n_tiles);
int pair_plan_fill(dram_conv_plan *pl);
int pair_plan_run(const dram_conv_plan *pl, int ctas, cudaStream_t st);

// plane-ring kernel (conv3d_slab.cu)
int slab_plan_supported(const dram_conv_desc *d);
int slab_plan_fill(dram_conv_plan *pl, const dram_conv_desc *d, const void *src1, const void *src2,
                   const void *weight, const EpiParams &epi);
int slab_plan_run(const dram_conv_plan *pl, int ctas, cudaStream_t st, const int *items, const int *count);
int slab_plan_listable(const dram_conv_plan *pl);
int slab_plan_worklist(const dram_conv_plan *pl, const uint32_t *bits, int radius, uint8_t *flags, int *list, int *count,
                       cudaStream_t st);

}  // namespace dram

using namespace dram;

extern "C" int dram_conv3d_out_dims(const dram_conv_desc *d, int32_t *dout, int32_t *hout,
                                    int32_t *wout) {
  DRAM_REQUIRE(d && dout && hout && wout, "dram_conv3d_out_dims: null argument");
  DRAM_REQUIRE(d->sd > 0 && d->sh > 0 && d->sw > 0, "dram_conv3d_out_dims: stride must be positive");
  *dout = conv_out(d->di, d->kd, d->sd, d->dd, d->pd);
  *hout = conv_out(d->hi, d->kh, d->sh, d->dh, d->ph);
  *wout = conv_out(d->wi, d->kw, d->sw, d->dw, d->pw);
  return DRAM_OK;
}

template <int BN, bool STAGED>
static int set_smem_attr() {
  return check_cuda(cudaFuncSetAttribute(conv3d_umma_kernel<BN, STAGED>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         ConvCfg<BN, STAGED>::SMEM_BYTES),
                    "cudaFuncSetAttribute(conv3d_umma_kernel)");
}
template <int BN, bool STAGED>
static int fill_tile_cfg(dram_conv_plan *pl) {
  pl->stages = ConvCfg<BN, STAGED>::STAGES;
  pl->smem_bytes = ConvCfg<BN, STAGED>::SMEM_BYTES;
  return set_smem_attr<BN, STAGED>();
}
template <int BN, bool STAGED>
static void launch_tiles(const dram_conv_plan *pl, dim3 grid, cudaStream_t st) {
  ConvKParams kp = pl->p;
  kp.epi = with_sat_counter(kp.epi);
  conv3d_umma_kernel<BN, STAGED><<<grid, STAGED ? NUM_THREADS_STAGED : NUM_THREADS, pl->smem_bytes, st>>>(
      pl->map_a1, pl->map_a2, pl->map_w, pl->map_out, pl->map_res, kp);
}

extern "C" int dram_conv3d_plan_create(const dram_conv_desc *d, const void *src1, const void *src2,
                                       const void *weight, const float *bias, const float *scale,
                                       const void *residual, void *out, const float *head_w,
                                       const float *head_b, float *head_out0, float *head_out1,
                                       dram_conv_plan **plan) {
  DRAM_REQUIRE(d && plan, "dram_conv3d_plan_create: null descriptor or plan pointer");
  *plan = nullptr;
  DRAM_REQUIRE(src1 && weight && bias, "dram_conv3d_plan_create: src1, weight and bias are required");
  DRAM_REQUIRE(d->n > 0 && d->di > 0 && d->hi > 0 && d->wi > 0, "conv3d: empty input");
  DRAM_REQUIRE(d->c1 > 0 && d->c1 % 64 == 0, "conv3d: c1=%d must be a positive multiple of 64", d->c1);
  DRAM_REQUIRE(d->c2 >= 0 && d->c2 % 64 == 0, "conv3d: c2=%d must be a multiple of 64", d->c2);
  DRAM_REQUIRE((d->c2 == 0) == (src2 == nullptr), "conv3d: src2 must be given exactly when c2 > 0");
  DRAM_REQUIRE(d->cout > 0 && d->cout % 32 == 0, "conv3d: cout=%d must be a multiple of 32", d->cout);
  DRAM_REQUIRE(d->kd >= 1 && d->kh >= 1 && d->kw >= 1 && d->kd <= 7 && d->kh <= 7 && d->kw <= 7,
               "conv3d: filter extent must be in 1..7");
  DRAM_REQUIRE(d->sd >= 1 && d->sh >= 1 && d->sw >= 1 && d->sd <= 8 && d->sh <= 8 && d->sw <= 8,
               "conv3d: stride must be in 1..8");
  DRAM_REQUIRE(d->dd >= 1 && d->dh >= 1 && d->dw >= 1, "conv3d: dilation must be >= 1");
  DRAM_REQUIRE(d->pd >= 0 && d->ph >= 0 && d->pw >= 0, "conv3d: padding must be >= 0");
  DRAM_REQUIRE(d->dtype == DRAM_DTYPE_BF16 || d->dtype == DRAM_DTYPE_F16, "conv3d: dtype must be bf16 (0) or fp16 (1)");
  DRAM_REQUIRE(d->algo >= DRAM_CONV_ALGO_AUTO && d->algo <= DRAM_CONV_ALGO_PLANES, "conv3d: bad algo %d", d->algo);
  DRAM_REQUIRE(d->epilogue >= DRAM_CONV_EPILOGUE_AUTO && d->epilogue <= DRAM_CONV_EPILOGUE_STAGED, "conv3d: bad epilogue %d",
               d->epilogue);
  DRAM_REQUIRE(d->store_out == 0 || out != nullptr, "conv3d: out is required when store_out != 0");
  DRAM_REQUIRE(d->store_out != 0 || d->n_heads > 0, "conv3d: nothing to write");

  int Do, Ho, Wo;
  dram_conv3d_out_dims(d, &Do, &Ho, &Wo);
  DRAM_REQUIRE(Do > 0 && Ho > 0 && Wo > 0, "conv3d: empty output");

  int block_n;
  if (d->cout % 256 == 0) block_n = 256;
  else if (d->cout % 128 == 0) block_n = 128;
  else if (d->cout % 64 == 0) block_n = 64;
  else block_n = 32;
  if (d->cout == 32) block_n = 32;
  DRAM_REQUIRE(d->cout % block_n == 0, "conv3d: cout=%d is not tileable", d->cout);

  if (d->n_heads > 0) {
    DRAM_REQUIRE(d->cout == 32, "conv3d: fused heads need cout == 32 (got %d)", d->cout);
    DRAM_REQUIRE(d->n_heads <= 2 && head_w && head_b && head_out0, "conv3d: bad head arguments");
    DRAM_REQUIRE(d->head_ch[0] >= 1 && (d->n_heads == 1 || (d->head_ch[1] >= 1 && head_out1)),
                 "conv3d: bad head channel counts");
    DRAM_REQUIRE(d->head_ch[0] + (d->n_heads == 2 ? d->head_ch[1] : 0) <= 16,
                 "conv3d: at most 16 head channels");
  }
  if (d->res_c > 0) {
    DRAM_REQUIRE(residual != nullptr, "conv3d: res_c > 0 but residual is NULL");
    DRAM_REQUIRE(d->res_c % 32 == 0 && d->res_c <= d->cout, "conv3d: res_c=%d must be a multiple of 32 and <= cout", d->res_c);
    DRAM_REQUIRE(d->res_stride >= 1, "conv3d: res_stride must be >= 1");
    DRAM_REQUIRE((Do - 1) * d->res_stride < d->res_d && (Ho - 1) * d->res_stride < d->res_h &&
                     (Wo - 1) * d->res_stride < d->res_w,
                 "conv3d: residual tensor %dx%dx%d too small for output %dx%dx%d at stride %d",
                 d->res_d, d->res_h, d->res_w, Do, Ho, Wo, d->res_stride);
  }

  EpiParams epi;
  memset(&epi, 0, sizeof(epi));
  epi.Do = Do; epi.Ho = Ho; epi.Wo = Wo;
  epi.cout = d->cout;
  epi.relu = d->relu;
  epi.is_f16 = d->dtype == DRAM_DTYPE_F16;
  epi.bias = bias;
  epi.scale = scale;
  epi.out = reinterpret_cast<uint16_t *>(out);
  epi.res = d->res_c > 0 ? reinterpret_cast<const uint16_t *>(residual) : nullptr;
  epi.res_c = d->res_c; epi.res_stride = d->res_stride > 0 ? d->res_stride : 1;
  epi.res_d = d->res_d; epi.res_h = d->res_h; epi.res_w = d->res_w;
  epi.n_heads = d->n_heads;
  epi.head_ch0 = d->n_heads > 0 ? d->head_ch[0] : 0;
  epi.head_ch1 = d->n_heads > 1 ? d->head_ch[1] : 0;
  epi.head_sigmoid = d->head_sigmoid;
  epi.store_out = d->store_out;
  epi.head_w = head_w; epi.head_b = head_b; epi.head_out0 = head_out0; epi.head_out1 = head_out1;

  const int taps = d->kd * d->kh * d->kw;
  const int64_t ktot = (int64_t)taps * (d->c1 + d->c2);

  dram_conv_plan *pl = new dram_conv_plan();
  memset(pl, 0, sizeof(*pl));
  pl->flops = 2LL * d->n * Do * Ho * Wo * (int64_t)d->cout * ktot;
  pl->block_n = block_n;

  // ---- plane-ring kernel for 3x3x3 / stride 1 / dilation 1 / Cout <= 64 ----------------------
  const bool want_planes = d->algo == DRAM_CONV_ALGO_PLANES ||
                           (d->algo == DRAM_CONV_ALGO_AUTO && d->tw == 0 && slab_plan_supported(d));
  if (d->src1_up2x && !(want_planes && slab_plan_supported(d))) {
    delete pl;
    set_error("conv3d: src1_up2x is implemented by the plane-ring kernel only (3x3x3, stride 1, dilation 1, cout 64)");
    return DRAM_E_ARG;
  }
  if (want_planes) {
    if (!slab_plan_supported(d)) {
      delete pl;
      set_error("conv3d: DRAM_CONV_ALGO_PLANES needs a 3x3x3 stride-1 dilation-1 pad-1 filter and cout of 32 or 64");
      return DRAM_E_ARG;
    }
    int rc = slab_plan_fill(pl, d, src1, src2, weight, epi);
    if (rc != DRAM_OK) {
      delete pl;
      return rc;
    }
    *plan = pl;
    return DRAM_OK;
  }

  // ---- per-tap TMA tile kernel ------------------------------------------------------------------
  // Tile shape: caller's choice or the candidate with the fewest tiles.
  int tw = d->tw, th = d->th, td = d->td;
  if (tw == 0 || th == 0 || td == 0) {
    static const int cand[][3] = {{8, 4, 4}, {4, 8, 4}, {4, 4, 8}, {8, 8, 2},  {8, 2, 8}, {2, 8, 8},
                                  {16, 4, 2}, {4, 16, 2}, {16, 2, 4}, {2, 16, 4}, {16, 8, 1}, {8, 16, 1},
                                  {32, 4, 1}, {4, 32, 1}, {32, 2, 2}, {16, 1, 8}, {128, 1, 1}};
    int64_t best = -1;
    for (auto &c : cand) {
      int64_t tiles = (int64_t)ceil_div(Wo, c[0]) * ceil_div(Ho, c[1]) * ceil_div(Do, c[2]);
      if (best < 0 || tiles < best) {
        best = tiles;
        tw = c[0];
        th = c[1];
        td = c[2];
      }
    }
  }
  if (!(is_pow2(tw) && is_pow2(th) && is_pow2(td) && tw * th * td == BLOCK_M)) {
    delete pl;
    set_error("conv3d: tile %dx%dx%d must be powers of two with product 128", tw, th, td);
    return DRAM_E_ARG;
  }
  if (!((tw - 1) * d->sw + 1 <= 256 && (th - 1) * d->sh + 1 <= 256 && (td - 1) * d->sd + 1 <= 256)) {
    delete pl;
    set_error("conv3d: TMA box too large for tile/stride");
    return DRAM_E_ARG;
  }

  pl->kind = 0;
  ConvKParams &p = pl->p;
  p.n = d->n; p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.Di = d->di; p.Hi = d->hi; p.Wi = d->wi;
  p.tw = tw; p.th = th; p.td = td; p.tw_log2 = ilog2(tw); p.th_log2 = ilog2(th);
  p.tiles_w = ceil_div(Wo, tw); p.tiles_h = ceil_div(Ho, th); p.tiles_d = ceil_div(Do, td);
  p.tiles_per_sample = p.tiles_w * p.tiles_h * p.tiles_d;
  p.num_n_tiles = d->cout / block_n;
  int64_t total = (int64_t)p.tiles_per_sample * d->n * p.num_n_tiles;
  if (total > 0x7fffffffLL) {
    delete pl;
    set_error("conv3d: too many tiles");
    return DRAM_E_ARG;
  }
  p.total_tiles = (int)total;
  p.kd = d->kd; p.kh = d->kh; p.kw = d->kw; p.sd = d->sd; p.sh = d->sh; p.sw = d->sw;
  p.dd = d->dd; p.dh = d->dh; p.dw = d->dw; p.pd = d->pd; p.ph = d->ph; p.pw = d->pw;
  p.chunks1 = d->c1 / BLOCK_K;
  p.chunks_total = (d->c1 + d->c2) / BLOCK_K;
  p.epi = epi;
  pl->m_tiles = p.tiles_per_sample * d->n;
  pl->n_tiles = p.num_n_tiles;

  int rc = encode_act_map(&pl->map_a1, src1, d->n, d->di, d->hi, d->wi, d->c1, BLOCK_K, tw, th, td, d->sw,
                          d->sh, d->sd, epi.is_f16);
  if (rc == DRAM_OK) {
    if (d->c2 > 0)
      rc = encode_act_map(&pl->map_a2, src2, d->n, d->di, d->hi, d->wi, d->c2, BLOCK_K, tw, th, td, d->sw,
                          d->sh, d->sd, epi.is_f16);
    else
      pl->map_a2 = pl->map_a1;
  }
  if (rc == DRAM_OK) rc = encode_weight_map(&pl->map_w, weight, d->cout, ktot, block_n, epi.is_f16);
  // Staged (shared memory + TMA) epilogue for the 1x1x1 convolutions: they are bound by the epilogue's global
  // accesses, which the direct path issues as one 16-byte access per lane and row.
  // The residual tile is a TMA box too: shortcut type A (fewer channels, strided read) falls out of the tensor
  // map — channel groups beyond res_c are out of bounds and arrive as zeros, the stride is the map's element stride.
  const bool res_tma = d->res_c % 64 == 0;
  const char *stg = getenv("DRAM_B200_STAGED_EPILOGUE");
  const bool staged_ok = taps == 1 && block_n >= 64 && d->store_out && d->n_heads == 0 && (d->res_c == 0 || res_tma);
  if (d->epilogue == DRAM_CONV_EPILOGUE_STAGED && !staged_ok) {
    delete pl;
    set_error("conv3d: the staged epilogue needs a 1x1x1 filter, cout %% 64 == 0, a stored output, no heads and res_c %% 64 == 0");
    return DRAM_E_ARG;
  }
  pl->staged = staged_ok && d->epilogue != DRAM_CONV_EPILOGUE_DIRECT &&
               (d->epilogue == DRAM_CONV_EPILOGUE_STAGED || !(stg && atoi(stg) == 0));
  // BLOCK_N = 256 staged exists without residual tiles only, and only on request (DRAM_CONV_EPILOGUE_STAGED): AUTO keeps
  // the N = 128 tiling that the bottleneck blocks were tuned with
  const bool staged256 = pl->staged && block_n == 256 && d->res_c == 0 && d->epilogue == DRAM_CONV_EPILOGUE_STAGED;
  if (pl->staged && block_n > 128 && !staged256) {  // re-tile N: the staged configuration with residual tiles holds BLOCK_N <= 128
    block_n = 128;
    pl->block_n = block_n;
    p.num_n_tiles = d->cout / block_n;
    const int64_t total2 = (int64_t)p.tiles_per_sample * d->n * p.num_n_tiles;
    if (total2 > 0x7fffffffLL) {
      delete pl;
      set_error("conv3d: too many tiles");
      return DRAM_E_ARG;
    }
    p.total_tiles = (int)total2;
    pl->n_tiles = p.num_n_tiles;
    rc = rc == DRAM_OK ? encode_weight_map(&pl->map_w, weight, d->cout, ktot, block_n, epi.is_f16) : rc;
  }
  p.staged_res = pl->staged && d->res_c > 0;
  pl->map_out = pl->map_a1;
  pl->map_res = pl->map_a1;
  if (rc == DRAM_OK && pl->staged) {
    // the staged epilogue moves quarter tiles: 32 consecutive rows of the tw x th x td brick (w fastest) are a box too
    const int qbw = tw < 32 ? tw : 32, qbh = (32 / qbw) < th ? 32 / qbw : th, qbd = 32 / (qbw * qbh);
    rc = encode_act_map(&pl->map_out, out, d->n, Do, Ho, Wo, d->cout, 64, qbw, qbh, qbd, 1, 1, 1, epi.is_f16);
    if (rc == DRAM_OK && p.staged_res)
      rc = encode_act_map(&pl->map_res, residual, d->n, d->res_d, d->res_h, d->res_w, d->res_c, 64, qbw, qbh, qbd,
                          epi.res_stride, epi.res_stride, epi.res_stride, epi.is_f16);
  }
  if (rc == DRAM_OK) {
    if (pl->staged) {
      switch (block_n) {
        case 64: rc = fill_tile_cfg<64, true>(pl); break;
        case 256: rc = fill_tile_cfg<256, true>(pl); break;
        default: rc = fill_tile_cfg<128, true>(pl); break;
      }
    } else if (d->tw == 0 && pair_plan_wanted(d, block_n, (int64_t)taps * p.chunks_total, pl->m_tiles, pl->n_tiles)) {
      rc = pair_plan_fill(pl);
    } else {
      switch (block_n) {
        case 32: rc = fill_tile_cfg<32, false>(pl); break;
        case 64: rc = fill_tile_cfg<64, false>(pl); break;
        case 128: rc = fill_tile_cfg<128, false>(pl); break;
        default: rc = fill_tile_cfg<256, false>(pl); break;
      }
    }
  }
  if (rc != DRAM_OK) {
    delete pl;
    return rc;
  }
  *plan = pl;
  return DRAM_OK;
}

extern "C" int dram_conv3d_plan_destroy(dram_conv_plan *plan) {
  delete plan;
  return DRAM_OK;
}

extern "C" int dram_conv3d_plan_info(const dram_conv_plan *plan, int64_t *flops, int32_t *m_tiles,
                                     int32_t *n_tiles, int32_t *block_n, int32_t *stages) {
  DRAM_REQUIRE(plan, "dram_conv3d_plan_info: null plan");
  if (flops) *flops = plan->flops;
  if (m_tiles) *m_tiles = plan->m_tiles;
  if (n_tiles) *n_tiles = plan->n_tiles;
  if (block_n) *block_n = plan->block_n;
  if (stages) *stages = plan->kind == 1 ? -plan->stages : plan->stages;  // negative: plane-ring kernel
  return DRAM_OK;
}

// What the kernels actually issue to the tensor pipe: full 128-voxel tiles (border tiles are padded), every
// non-skipped (tap, chunk) stage at the plan's BLOCK_N — i.e. the algorithmic 2*M*N*K minus the taps skipped in the
// zero padding plus the tile-quantisation padding.
static bool host_tap_is_padding(int i0, int extent, int stride, int in_size) {
  return (i0 + (extent - 1) * stride < 0) || (i0 >= in_size);
}
static bool host_brick_tap_skipped(const ConvKParams &p, int m_tile, int zd, int zh, int zw) {
  const int r = m_tile % p.tiles_per_sample;
  const int iw = r % p.tiles_w, r2 = r / p.tiles_w, ih = r2 % p.tiles_h, id = r2 / p.tiles_h;
  return host_tap_is_padding(id * p.td * p.sd + zd * p.dd - p.pd, p.td, p.sd, p.Di) ||
         host_tap_is_padding(ih * p.th * p.sh + zh * p.dh - p.ph, p.th, p.sh, p.Hi) ||
         host_tap_is_padding(iw * p.tw * p.sw + zw * p.dw - p.pw, p.tw, p.sw, p.Wi);
}

extern "C" int dram_conv3d_plan_executed_flops(const dram_conv_plan *plan, int64_t *flops) {
  DRAM_REQUIRE(plan && flops, "dram_conv3d_plan_executed_flops: null argument");
  if (plan->kind == 1) {  // plane ring: every item issues 4 planes x 27 taps x all chunks, N = cout
    const SlabParams &sp = plan->sp;
    if (sp.stream) {  // every (output plane, kd) pair inside the volume is one N = 32 block of 9 x 4 MMAs; no D padding
      const int64_t cols = (int64_t)sp.n * sp.cols_w * sp.cols_h;
      *flops = 2LL * cols * (3LL * sp.D - 2) * 128 * 32 * 9 * 64;
      return DRAM_OK;
    }
    const int group = plan->block_n == 128 ? 2 : 4;  // output planes per item (conv3d_slab.cu slab_group)
    *flops = 2LL * sp.items_total * group * 128 * (int64_t)plan->block_n * 27 * sp.chunks_total * 64;
    return DRAM_OK;
  }
  const ConvKParams &p = plan->p;
  const int m_tiles = plan->m_tiles;
  int64_t stages = 0;  // (brick, tap) pairs issued, per n-tile
  if (plan->pair) {
    for (int pr = 0; 2 * pr < m_tiles; ++pr)
      for (int zd = 0; zd < p.kd; ++zd)
        for (int zh = 0; zh < p.kh; ++zh)
          for (int zw = 0; zw < p.kw; ++zw) {
            const bool s0 = host_brick_tap_skipped(p, 2 * pr, zd, zh, zw);
            const bool s1 = 2 * pr + 1 < m_tiles ? host_brick_tap_skipped(p, 2 * pr + 1, zd, zh, zw) : true;
            if (!(s0 && s1)) stages += 2;  // both bricks run the MMA when either needs the tap
          }
  } else {
    for (int m = 0; m < m_tiles; ++m)
      for (int zd = 0; zd < p.kd; ++zd)
        for (int zh = 0; zh < p.kh; ++zh)
          for (int zw = 0; zw < p.kw; ++zw)
            if (!host_brick_tap_skipped(p, m, zd, zh, zw)) ++stages;
  }
  *flops = 2LL * stages * p.num_n_tiles * 128 * (int64_t)plan->block_n * p.chunks_total * 64;
  return DRAM_OK;
}

extern "C" int dram_conv3d_run(const dram_conv_plan *plan, int32_t max_ctas, void *stream) {
  DRAM_REQUIRE(plan, "dram_conv3d_run: null plan");
  int ctas = sm_count();
  if (max_ctas > 0 && max_ctas < ctas) ctas = max_ctas;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (plan->kind == 1) return slab_plan_run(plan, ctas, st, nullptr, nullptr);
  if (plan->pair) return pair_plan_run(plan, ctas, st);
  if (plan->p.total_tiles < ctas) ctas = plan->p.total_tiles;
  dim3 grid(ctas);
  if (plan->staged) {
    switch (plan->block_n) {
      case 64: launch_tiles<64, true>(plan, grid, st); break;
      case 256: launch_tiles<256, true>(plan, grid, st); break;
      default: launch_tiles<128, true>(plan, grid, st); break;
    }
  } else {
    switch (plan->block_n) {
      case 32: launch_tiles<32, false>(plan, grid, st); break;
      case 64: launch_tiles<64, false>(plan, grid, st); break;
      case 128: launch_tiles<128, false>(plan, grid, st); break;
      default: launch_tiles<256, false>(plan, grid, st); break;
    }
  }
  DRAM_CHECK_LAUNCH("conv3d_umma_kernel launch");
  return DRAM_OK;
}

static bool conv_listable(const dram_conv_plan *plan) { return plan->kind == 1 && slab_plan_listable(plan); }

extern "C" int dram_conv3d_worklist_size(const dram_conv_plan *plan, int32_t *entries) {
  DRAM_REQUIRE(plan && entries, "dram_conv3d_worklist_size: null argument");
  *entries = conv_listable(plan) ? (plan->sp.stream ? plan->sp.steps_total : plan->sp.items_total) : 0;
  return DRAM_OK;
}

extern "C" int dram_conv3d_worklist(const dram_conv_plan *plan, const uint32_t *support, int32_t radius, uint8_t *flags,
                                    int32_t *items, int32_t *count, void *stream) {
  DRAM_REQUIRE(plan, "dram_conv3d_worklist: null plan");
  DRAM_REQUIRE(conv_listable(plan), "dram_conv3d_worklist: this plan's kernel takes no work list");
  return slab_plan_worklist(plan, support, radius, flags, items, count, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int dram_conv3d_run_listed(const dram_conv_plan *plan, const int32_t *items, const int32_t *count,
                                      int32_t max_ctas, void *stream) {
  DRAM_REQUIRE(plan && items && count, "dram_conv3d_run_listed: null argument");
  DRAM_REQUIRE(conv_listable(plan), "dram_conv3d_run_listed: this plan's kernel takes no work list");
  int ctas = sm_count();
  if (max_ctas > 0 && max_ctas < ctas) ctas = max_ctas;
  return slab_plan_run(plan, ctas, reinterpret_cast<cudaStream_t>(stream), items, count);
}
