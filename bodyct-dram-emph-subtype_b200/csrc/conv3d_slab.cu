// K1, plane-ring variant — 3x3x3 / stride 1 / dilation 1 / pad 1 convolutions with Cout of 32 or 64
// (layer1, the whole decoder).
//
// Why: with one TMA box per (tap, chunk) every 128-clock MMA chunk ingests a 16 KiB activation tile and an
// 8 KiB weight tile, ~190 B/clk/SM against the ~36 B/clk/SM the L2->SM fabric sustains
// (profiles/conv_ncu_r1.md).  Here
//   * the CTA owns a column of the volume, 8 (W) x 16 (H) voxels wide, and marches along D;
//   * every input plane of the column (10 x 18 voxels with halo, 64 channels = 23 KiB) is fetched ONCE by
//     one TMA box into a shared-memory ring; zero padding = TMA out-of-bounds fill;
//   * an output tile is one 8 x 16 slab (128 voxels); its A operand for tap (kd,kh,kw) is the plane
//     d+kd-1 viewed through a UMMA descriptor whose start address is shifted by (kh*10+kw) rows and whose
//     8-row-group stride (SBO) is the plane pitch 10*128 B — no data is moved per tap;
//   * four consecutive output planes accumulate side by side in TMEM (two sets of 4 x N columns);
//   * kd is stacked along the MMA's N dimension: with Cout <= 64 the tensor pipe is bound by the
//     shared-memory read of the A operand (4 KiB per M128 x N64 x K16 MMA = the full 128 B/clk; ncu:
//     l1tex__data_pipe_tc_wavefronts_mem_shared 72 %, profiles/aux_ncu_r1d.md).  Input plane j of an item
//     contributes to output planes j, j-1, j-2 through kd = 0, 1, 2, and those accumulators sit in adjacent
//     TMEM columns, so ONE MMA with B = [W(kd=2); W(kd=1); W(kd=0)] (N = 3*Cout) replaces three: the A
//     tile is read once for up to 192 output channels.  A weight stage therefore holds the three kd taps
//     of one (kh,kw).
//
//   * UP variant (decoder stages us1.0 / us2.0, med3d.py:83-89): source 1 is given at HALF resolution and
//     the x2 trilinear (align_corners=True) up-sampling happens inside the kernel: the low-resolution
//     patch under a plane (<= 11 x 7 voxels x 64 channels per source plane) streams through a small TMA
//     ring, four extra warps interpolate it into the plane slot in the SWIZZLE_128B layout with the very
//     arithmetic of K4 (bit-identical values), and the up-sampled tensor is never written to HBM.
//
// Roles (224 threads; UP: 352): warps 0-3 epilogue, warp 4 lane 0 plane producer, warp 5 MMA issuer (owns TMEM),
// warp 6 lane 0 weight producer, UP: warps 7-10 interpolate.  Work items = (column, group of 4 planes); every CTA takes a
// contiguous range of items (D fastest), so consecutive groups of a column reuse two resident planes.
#include <string.h>

#include "conv_plan.h"

namespace dram {

static constexpr int SL_W = 8, SL_H = 16;                    // slab = 8 x 16 voxels
// Output planes per work item: 4 for Cout 32 / 64; 2 for Cout 128 (TMEM holds 2 x GROUP x Cout fp32 columns = 512, and
// with two output planes a plane feeds at most two of them, so the kd-stacked N stays <= 256).
__host__ __device__ constexpr int slab_group(int block_n) { return block_n == 128 ? 2 : 4; }
static constexpr int PL_W = SL_W + 2, PL_H = SL_H + 2;       // input plane with halo
static constexpr int PLANE_BYTES = PL_W * PL_H * 128;        // 23040
static constexpr int PLANE_PITCH = 23 * 1024;                // slot pitch, 1 KiB aligned for SWIZZLE_128B
#ifndef DRAM_SLAB_RING
#define DRAM_SLAB_RING 7
#endif
static constexpr int RING = DRAM_SLAB_RING;
static constexpr int RING_UP = 6;                            // plane slots of the UP variant
static constexpr int LP_W = 7, LP_H = 11;                    // low-resolution patch under a 10 x 18 plane
static constexpr int LP_BYTES = LP_W * LP_H * 128;           // 9856
static constexpr int LP_PITCH = 10 * 1024;
static constexpr int LP_RING = 3;
static constexpr int UP_WARP0 = 7, UP_THREADS = 128;
static constexpr int SL_THREADS = 224;
static constexpr int SL_A_WARP = 4, SL_MMA_WARP = 5, SL_B_WARP = 6;
static constexpr int SL_BLOCK_K = 64;

template <int BLOCK_N, bool UP = false>
struct SlabCfg {
  static constexpr int GROUP = slab_group(BLOCK_N);
  static constexpr int ITEM_PLANES = GROUP + 2;             // input planes that feed GROUP output planes
  static constexpr int MAX_BLK = GROUP < 3 ? GROUP : 3;     // output planes one input plane feeds (kd stacked along N)
  static constexpr int RING_ = UP ? RING_UP : (BLOCK_N == 128 ? 5 : RING);
  static constexpr int THREADS = UP ? SL_THREADS + UP_THREADS : SL_THREADS;
  static constexpr int B_BLOCK_BYTES = BLOCK_N * 128;       // one tap: Cout rows x 64 channels
  static constexpr int B_STAGE_BYTES = 3 * B_BLOCK_BYTES;   // [kd=2; kd=1; kd=0] of one (kh,kw)
#ifndef DRAM_SLAB_BSTAGES64
#define DRAM_SLAB_BSTAGES64 2
#endif
  static constexpr int B_STAGES = BLOCK_N == 64 ? DRAM_SLAB_BSTAGES64 : (BLOCK_N == 128 ? 2 : 4);
  static constexpr int TMEM_COLS = 2 * GROUP * BLOCK_N;     // 512 (N = 64, 128) / 256 (N = 32)
  static constexpr int LP_TOTAL = UP ? LP_RING * LP_PITCH : 0;
  static constexpr int SMEM_BYTES = 1024 + RING_ * PLANE_PITCH + B_STAGES * B_STAGE_BYTES + LP_TOTAL + 256;
};

struct SlabItem {
  int sample, w0, h0, q0, g;
};
__device__ __forceinline__ SlabItem decode_item(const SlabParams &p, int item, int group) {
  SlabItem it;
  const int col = item / p.groups_d;
  it.g = item - col * p.groups_d;
  it.q0 = it.g * group;
  const int per_sample = p.cols_w * p.cols_h;
  it.sample = col / per_sample;
  const int r = col - it.sample * per_sample;
  const int ih = r / p.cols_w;
  it.w0 = (r - ih * p.cols_w) * SL_W;
  it.h0 = ih * SL_H;
  return it;
}

// K-major SWIZZLE_128B descriptor with an arbitrary (16-byte aligned) start and 8-row-group stride.
__device__ __forceinline__ uint64_t make_sw128_desc_sbo(uint32_t smem_addr, uint32_t sbo_bytes, int base_offset_mode) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  if (base_offset_mode) d |= (uint64_t)((smem_addr >> 7) & 7) << 49;
  d |= (uint64_t)2 << 61;
  return d;
}

// Low-resolution source range [lo, hi] that the output range [o_lo, o_hi] (clipped to the tensor) reads.
__device__ __forceinline__ int up_src_lo(int o_lo, float scale, int in_size) {
  return lin_index_ac(o_lo < 0 ? 0 : o_lo, scale, in_size).i0;
}
__device__ __forceinline__ int up_src_hi(int o_hi, int out_size, float scale, int in_size) {
  return lin_index_ac(o_hi > out_size - 1 ? out_size - 1 : o_hi, scale, in_size).i1;
}

template <int BLOCK_N, bool UP>
__global__ void __launch_bounds__((SlabCfg<BLOCK_N, UP>::THREADS), 1)
conv3d_slab_kernel(const __grid_constant__ CUtensorMap map_a1, const __grid_constant__ CUtensorMap map_a2,
                   const __grid_constant__ CUtensorMap map_w, const __grid_constant__ SlabParams p) {
  using Cfg = SlabCfg<BLOCK_N, UP>;
  constexpr int B_STAGES = Cfg::B_STAGES;
  constexpr int RING = Cfg::RING_;  // shadows the namespace constant
  constexpr int SL_GROUP = Cfg::GROUP, ITEM_PLANES = Cfg::ITEM_PLANES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_base = smem_base + RING * PLANE_PITCH;
  const uint32_t bar_base = b_base + B_STAGES * Cfg::B_STAGE_BYTES;
  auto plane_addr = [&](int s) { return smem_base + (uint32_t)s * PLANE_PITCH; };
  auto plane_full = [&](int s) { return bar_base + 8u * s; };
  auto plane_empty = [&](int s) { return bar_base + 8u * (RING + s); };
  auto b_addr = [&](int s) { return b_base + (uint32_t)s * Cfg::B_STAGE_BYTES; };
  auto b_full = [&](int s) { return bar_base + 8u * (2 * RING + s); };
  auto b_empty = [&](int s) { return bar_base + 8u * (2 * RING + B_STAGES + s); };
  auto tmem_full = [&](int a) { return bar_base + 8u * (2 * RING + 2 * B_STAGES + a); };
  auto tmem_empty = [&](int a) { return bar_base + 8u * (2 * RING + 2 * B_STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * RING + 2 * B_STAGES + 4);
  // UP only: low-resolution plane ring behind the barriers' 256-byte block
  const uint32_t lp_base = bar_base + 256u;
  auto lp_addr = [&](int s) { return lp_base + (uint32_t)s * LP_PITCH; };
  auto lp_full = [&](int s) { return bar_base + 8u * (2 * RING + 2 * B_STAGES + 5 + s); };
  auto lp_empty = [&](int s) { return bar_base + 8u * (2 * RING + 2 * B_STAGES + 5 + LP_RING + s); };

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < RING; ++s) {
      mbar_init(plane_full(s), 1);
      mbar_init(plane_empty(s), 1);
    }
    for (int s = 0; s < B_STAGES; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(b_empty(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full(a), 1);
      mbar_init(tmem_empty(a), 128);
    }
    if (UP)
      for (int s = 0; s < LP_RING; ++s) {
        mbar_init(lp_full(s), 1);
        mbar_init(lp_empty(s), UP_THREADS);
      }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == SL_MMA_WARP) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  if (warp == SL_A_WARP && lane == 0) {
    prefetch_tensormap(&map_a1);
    prefetch_tensormap(&map_a2);
  }
  if (warp == SL_B_WARP && lane == 0) prefetch_tensormap(&map_w);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);  // provably warp-uniform

  // contiguous, balanced range of work items (positions in the work list, if there is one) for this CTA
  const int items_total = p.items ? *p.count : p.items_total;
  const int item_begin = (int)(((long long)blockIdx.x * items_total) / gridDim.x);
  const int item_end = (int)(((long long)(blockIdx.x + 1) * items_total) / gridDim.x);
  auto item_at = [&](int i) { return p.items ? __ldg(p.items + i) : i; };
  const bool single_chunk = !UP && p.chunks_total == 1;  // UP layers never reuse planes across items

  if (warp == SL_A_WARP) {
    if (lane == 0) {
      unsigned seq_end = 0;
      unsigned lseq = 0;  // UP: running index of low-resolution planes through the LP ring
      int prev = -1;
      for (int i = item_begin; i < item_end; ++i) {
        const int item = item_at(i);
        const SlabItem it = decode_item(p, item, Cfg::GROUP);
        // two planes of the previous item are reused if it was the previous group of the same column
        const bool reuse = single_chunk && prev == item - 1 && it.g > 0;
        prev = item;
        for (int c = 0; c < p.chunks_total; ++c) {
          const unsigned seq_base = seq_end - (reuse ? 2u : 0u);
          seq_end = seq_base + ITEM_PLANES;
          if (UP && c < p.chunks1) {
            // the interpolating warps fill the plane slots of this chunk; feed them the low-resolution
            // planes under output planes q0-1 .. q0+4, in order
            const int zl0 = up_src_lo(it.q0 - 1, p.up_sd, p.Dl);
            const int zl1 = up_src_hi(it.q0 + SL_GROUP, p.D, p.up_sd, p.Dl);
            const int hl0 = up_src_lo(it.h0 - 1, p.up_sh, p.Hl), wl0 = up_src_lo(it.w0 - 1, p.up_sw, p.Wl);
            for (int zl = zl0; zl <= zl1; ++zl, ++lseq) {
              const int ls = lseq % LP_RING;
              mbar_wait(lp_empty(ls), ((lseq / LP_RING) & 1u) ^ 1u);
              mbar_expect_tx(lp_full(ls), LP_BYTES);
              tma_load_5d(lp_addr(ls), &map_a1, lp_full(ls), c * SL_BLOCK_K, wl0, hl0, zl, it.sample);
            }
            // The plane slots of this chunk are filled by the interpolating warps.  mbarrier waits only
            // tell phases apart by parity, so every agent that fills plane slots has to observe every
            // hand-back of every slot, or it could run two phases ahead and take a slot that is still in use.
            for (int j = 0; j < ITEM_PLANES; ++j) {
              const unsigned seq = seq_base + j;
              mbar_wait(plane_empty(seq % RING), ((seq / RING) & 1u) ^ 1u);
            }
            continue;
          }
          for (int j = reuse ? 2 : 0; j < ITEM_PLANES; ++j) {
            const unsigned seq = seq_base + j;
            const int slot = seq % RING;
            mbar_wait(plane_empty(slot), ((seq / RING) & 1u) ^ 1u);
            mbar_expect_tx(plane_full(slot), PLANE_BYTES);
            if (c < p.chunks1)
              tma_load_5d(plane_addr(slot), &map_a1, plane_full(slot), c * SL_BLOCK_K, it.w0 - 1, it.h0 - 1,
                          it.q0 - 1 + j, it.sample);
            else
              tma_load_5d(plane_addr(slot), &map_a2, plane_full(slot), (c - p.chunks1) * SL_BLOCK_K, it.w0 - 1,
                          it.h0 - 1, it.q0 - 1 + j, it.sample);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == SL_B_WARP) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int i = item_begin; i < item_end; ++i) {
        for (int c = 0; c < p.chunks_total; ++c) {
          for (int hw = 0; hw < 9; ++hw) {  // one stage = the three kd taps of (kh,kw), kd descending
            mbar_wait(b_empty(stage), phase ^ 1u);
            mbar_expect_tx(b_full(stage), Cfg::B_STAGE_BYTES);
#pragma unroll
            for (int blk = 0; blk < 3; ++blk) {
              const int tap = (2 - blk) * 9 + hw;
              tma_load_2d(b_addr(stage) + (uint32_t)(blk * Cfg::B_BLOCK_BYTES), &map_w, b_full(stage),
                          (tap * p.chunks_total + c) * SL_BLOCK_K, 0);
            }
            if (++stage == B_STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == SL_MMA_WARP) {
    {  // the whole warp walks the loops (uniform control flow); one elected lane issues.
      // The issuing thread is the bottleneck of this kernel if it spends more than ~30 instructions per MMA (a
      // single warp retires a dependent instruction every few clocks, an M128 x N64 x K16 MMA lasts 32-48): measured
      // in round 2, us3 (N = 32) took 90 % of the time of us2.1 (N = 64) — time followed the MMA COUNT, ~95 clocks
      // each.  So everything that does not change per MMA is hoisted: the plane descriptors are built once per
      // chunk (six 64-bit values, broadcast so that they live in uniform registers), the (kh, kw) / kd / K-step
      // offsets are compile-time constants of the fully unrolled loops, and a stage's 24 MMAs are issued from ONE
      // elected region: two 64-bit uniform adds per tcgen05.mma.
      uint32_t idesc[Cfg::MAX_BLK];
#pragma unroll
      for (int nb = 0; nb < Cfg::MAX_BLK; ++nb) idesc[nb] = make_idesc_16bit(128, (nb + 1) * BLOCK_N, p.epi.is_f16);
      const uint64_t desc_a_const = make_sw128_desc_sbo(0u, PL_W * 128, 0);
      const uint64_t desc_b_const = make_sw128_desc(0u);
      int stage = 0;
      uint32_t phase = 0;
      unsigned seq_end = 0;
      int buf = 0;
      uint32_t buf_phase = 0;
      int prev = -1;
      for (int i = item_begin; i < item_end; ++i) {
        const int item = item_at(i);
        const SlabItem it = decode_item(p, item, Cfg::GROUP);
        mbar_wait(tmem_empty(buf), buf_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t tmem_d0 = tmem_base + (uint32_t)(buf * SL_GROUP * BLOCK_N);
        // the same rule as the producer's: the next list entry is the next group of this column
        const bool reuse = single_chunk && prev == item - 1 && it.g > 0;
        const bool next_reuse = single_chunk && i + 1 < item_end && it.g + 1 < p.groups_d && item_at(i + 1) == item + 1;
        prev = item;
        for (int c = 0; c < p.chunks_total; ++c) {
          const unsigned seq_base = seq_end - (reuse ? 2u : 0u);
          seq_end = seq_base + ITEM_PLANES;
          // per-plane constants of this chunk: A descriptor of the slot base, barrier addresses / parities
          uint64_t da_plane[ITEM_PLANES];
          uint32_t full_bar[ITEM_PLANES], full_par[ITEM_PLANES], empty_bar[ITEM_PLANES];
#pragma unroll
          for (int j = 0; j < ITEM_PLANES; ++j) {
            const unsigned seq = seq_base + j;
            const int slot = seq % RING;
            uint32_t pa = plane_addr(slot);
            if (p.desc_base_offset_mode) pa |= 0u;  // (knob kept for the plan struct; the base-offset field stays 0)
            pa = __shfl_sync(0xffffffffu, pa, 0);   // provably warp-uniform -> uniform registers
            da_plane[j] = desc_a_const | (uint64_t)((pa & 0x3FFFFu) >> 4);
            full_bar[j] = plane_full(slot);
            full_par[j] = (seq / RING) & 1u;
            empty_bar[j] = plane_empty(slot);
          }
          const bool first_chunk = c == 0;
#pragma unroll
          for (int hw = 0; hw < 9; ++hw) {
            constexpr int kRowBytes = 128;
            const int kh = hw / 3, kw = hw - 3 * kh;                       // constants after unrolling
            const uint32_t row_off16 = (uint32_t)((kh * PL_W + kw) * kRowBytes) >> 4;
            mbar_wait(b_full(stage), phase);
            tcgen05_fence_after();
            uint32_t bb = b_addr(stage);
            bb = __shfl_sync(0xffffffffu, bb, 0);
            const uint64_t db_stage = desc_b_const | (uint64_t)((bb & 0x3FFFFu) >> 4);
            if (hw == 0) {
              // planes of this chunk arrive in order during its first stage: wait for each just before its MMAs
#pragma unroll
              for (int j = 0; j < ITEM_PLANES; ++j) {
                mbar_wait(full_bar[j], full_par[j]);
                tcgen05_fence_after();
                const int kd_hi = j < 2 ? j : 2, kd_lo = j > SL_GROUP - 1 ? j - (SL_GROUP - 1) : 0;
                const int nblk = kd_hi - kd_lo + 1, t_min = j - kd_hi;
                const uint64_t da = da_plane[j] + row_off16;
                const uint64_t db = db_stage + (uint64_t)(((2 - kd_hi) * Cfg::B_BLOCK_BYTES) >> 4);
                const uint32_t dcol = tmem_d0 + (uint32_t)(t_min * BLOCK_N);
                if (elect_one_sync()) {
                  if (first_chunk) {  // accumulators are initialised tile by tile: tile t's first touch is kd == 0
#pragma unroll
                    for (int q = 0; q < nblk; ++q) {
                      const uint64_t dbq = db + (uint64_t)((q * Cfg::B_BLOCK_BYTES) >> 4);
#pragma unroll
                      for (int k = 0; k < 4; ++k)
                        umma_bf16(dcol + (uint32_t)(q * BLOCK_N), da + (uint64_t)(2 * k), dbq + (uint64_t)(2 * k), idesc[0],
                                  (k > 0 || kd_hi - q > 0) ? 1u : 0u);
                    }
                  } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                      umma_bf16(dcol, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc[nblk - 1], 1u);
                  }
                }
                __syncwarp();
              }
              if (elect_one_sync()) umma_commit(b_empty(stage));
              __syncwarp();
            } else {
              if (elect_one_sync()) {
                // Issue order inside a stage (-DDRAM_SLAB_MMA_ORDER): 0 = plane by plane, the four K steps of a plane
                // back to back; 1 (default) = K steps outermost and the planes visited so that neighbouring
                // instructions write disjoint output tiles where possible (GROUP 4: plane j feeds tiles {j-2..j} & [0,3],
                // order 0,4,1,5,2,3 leaves only 2 -> 3 sharing columns; GROUP 2: 0,3,1,2).  Measured 2-3 % faster on the
                // 64-channel layers (profiles/convbench_order_r2e.log): back-to-back instructions on the same
                // accumulator columns serialise a little.  tcgen05.mma instructions of one thread execute in issue
                // order, so the accumulation order per output element is still fixed: results are reproducible bit for
                // bit (tests/test_conv3d_gpu.py::test_convolutions_are_reproducible_bit_for_bit, tools/train_repro_check.py)
                // — they differ from order 0 only in the last bits of the fp32 sums.
#ifndef DRAM_SLAB_MMA_ORDER
#define DRAM_SLAB_MMA_ORDER 1
#endif
                constexpr int kOrder4[6] = {0, 4, 1, 5, 2, 3};
                constexpr int kOrder2[4] = {0, 3, 1, 2};
#if DRAM_SLAB_MMA_ORDER == 0
#pragma unroll
                for (int j = 0; j < ITEM_PLANES; ++j) {
#pragma unroll
                  for (int k = 0; k < 4; ++k) {
#else
#pragma unroll
                for (int k = 0; k < 4; ++k) {
#pragma unroll
                  for (int jj = 0; jj < ITEM_PLANES; ++jj) {
                    const int j = SL_GROUP == 4 ? kOrder4[jj < 6 ? jj : 0] : kOrder2[jj < 4 ? jj : 0];
#endif
                    // input plane j feeds output tiles t = j - kd, kd = kd_hi .. kd_lo (descending kd = ascending t)
                    const int kd_hi = j < 2 ? j : 2, kd_lo = j > SL_GROUP - 1 ? j - (SL_GROUP - 1) : 0;
                    const int nblk = kd_hi - kd_lo + 1, t_min = j - kd_hi;
                    const uint64_t da = da_plane[j] + row_off16;
                    const uint64_t db = db_stage + (uint64_t)(((2 - kd_hi) * Cfg::B_BLOCK_BYTES) >> 4);
                    const uint32_t dcol = tmem_d0 + (uint32_t)(t_min * BLOCK_N);
                    umma_bf16(dcol, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc[nblk - 1], 1u);
                  }
                }
                // last stage of the chunk: hand the planes back (the commits track every MMA issued so far)
                if (hw == 8) {
#pragma unroll
                  for (int j = 0; j < ITEM_PLANES; ++j)
                    if (j < SL_GROUP || !next_reuse) umma_commit(empty_bar[j]);
                }
                umma_commit(b_empty(stage));
              }
              __syncwarp();
            }
            if (++stage == B_STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
        if (elect_one_sync()) umma_commit(tmem_full(buf));
        __syncwarp();
        if (++buf == 2) {
          buf = 0;
          buf_phase ^= 1u;
        }
      }
    }
    __syncwarp();
  } else if (UP && warp >= UP_WARP0) {
    // ------------------------------- UP: interpolating warps -------------------------------
    // Output plane z of the column = 18 x 10 voxel rows of 64 channels; a thread builds 16-byte chunks
    // (8 channels) of rows: trilinear of 8 low-resolution voxels read from the LP ring, same fp32 operation
    // order as K4, rounded once to the storage type, stored at the SWIZZLE_128B position the UMMA view expects.
    const int tid = threadIdx.x - UP_WARP0 * 32;
    const int is_f16 = p.epi.is_f16;
    unsigned seq_end = 0, lseq_base = 0;
    for (int i = item_begin; i < item_end; ++i) {
      const SlabItem it = decode_item(p, item_at(i), Cfg::GROUP);
      for (int c = 0; c < p.chunks_total; ++c) {
        const unsigned seq_base = seq_end;  // UP layers have more than one chunk: no plane reuse across items
        seq_end = seq_base + ITEM_PLANES;
        if (c >= p.chunks1) {  // TMA-filled chunk: only observe the hand-backs (see the producer)
          for (int j = 0; j < ITEM_PLANES; ++j) {
            const unsigned seq = seq_base + j;
            mbar_wait(plane_empty(seq % RING), ((seq / RING) & 1u) ^ 1u);
          }
          continue;
        }
        const int zl0 = up_src_lo(it.q0 - 1, p.up_sd, p.Dl);
        const int zl1 = up_src_hi(it.q0 + SL_GROUP, p.D, p.up_sd, p.Dl);
        const int hl0 = up_src_lo(it.h0 - 1, p.up_sh, p.Hl), wl0 = up_src_lo(it.w0 - 1, p.up_sw, p.Wl);
        int released = zl0;  // low-resolution planes below this index have been handed back
        for (int j = 0; j < ITEM_PLANES; ++j) {
          const unsigned seq = seq_base + j;
          const int slot = seq % RING;
          const int z = it.q0 - 1 + j;
          const bool zok = z >= 0 && z < p.D;
          mbar_wait(plane_empty(slot), ((seq / RING) & 1u) ^ 1u);
          LinIdx id = {0, 0, 0.0f, 0.0f};
          uint32_t lp0 = 0, lp1 = 0;
          if (zok) {
            id = lin_index_ac(z, p.up_sd, p.Dl);
            // planes below id.i0 are not read any more
            for (; released < id.i0; ++released) mbar_arrive(lp_empty((lseq_base + (unsigned)(released - zl0)) % LP_RING));
            const unsigned s0 = lseq_base + (unsigned)(id.i0 - zl0), s1 = lseq_base + (unsigned)(id.i1 - zl0);
            mbar_wait(lp_full(s0 % LP_RING), (s0 / LP_RING) & 1u);
            mbar_wait(lp_full(s1 % LP_RING), (s1 / LP_RING) & 1u);
            lp0 = lp_addr(s0 % LP_RING);
            lp1 = lp_addr(s1 % LP_RING);
          }
          const uint32_t dst0 = plane_addr(slot);
#pragma unroll 1
          for (int task = tid; task < PL_W * PL_H * 8; task += UP_THREADS) {
            const int r = task >> 3, c16 = task & 7;
            const int ph = r / PL_W, pw = r - ph * PL_W;
            const int oh = it.h0 - 1 + ph, ow = it.w0 - 1 + pw;
            uint32_t o[4] = {0u, 0u, 0u, 0u};
            if (zok && oh >= 0 && oh < p.H && ow >= 0 && ow < p.W) {
              const LinIdx ih = lin_index_ac(oh, p.up_sh, p.Hl), iw = lin_index_ac(ow, p.up_sw, p.Wl);
              const uint32_t o00 = (uint32_t)(((ih.i0 - hl0) * LP_W + (iw.i0 - wl0)) * 128 + c16 * 16);
              const uint32_t o01 = (uint32_t)(((ih.i0 - hl0) * LP_W + (iw.i1 - wl0)) * 128 + c16 * 16);
              const uint32_t o10 = (uint32_t)(((ih.i1 - hl0) * LP_W + (iw.i0 - wl0)) * 128 + c16 * 16);
              const uint32_t o11 = (uint32_t)(((ih.i1 - hl0) * LP_W + (iw.i1 - wl0)) * 128 + c16 * 16);
              uint32_t a0[4], b0[4], c0[4], d0[4], a1[4], b1[4], c1[4], d1[4];
              auto lds = [](uint32_t addr, uint32_t (&v)[4]) {
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
                             : "r"(addr));
              };
              lds(lp0 + o00, a0); lds(lp0 + o01, b0); lds(lp0 + o10, c0); lds(lp0 + o11, d0);
              lds(lp1 + o00, a1); lds(lp1 + o01, b1); lds(lp1 + o10, c1); lds(lp1 + o11, d1);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 fa0 = unpack2(a0[q], is_f16), fb0 = unpack2(b0[q], is_f16), fc0 = unpack2(c0[q], is_f16),
                             fd0 = unpack2(d0[q], is_f16);
                const float2 fa1 = unpack2(a1[q], is_f16), fb1 = unpack2(b1[q], is_f16), fc1 = unpack2(c1[q], is_f16),
                             fd1 = unpack2(d1[q], is_f16);
                const float x0 = bilerp_hw(fa0.x, fb0.x, fc0.x, fd0.x, iw.w0, iw.w1, ih.w0, ih.w1);
                const float x1 = bilerp_hw(fa1.x, fb1.x, fc1.x, fd1.x, iw.w0, iw.w1, ih.w0, ih.w1);
                const float y0 = bilerp_hw(fa0.y, fb0.y, fc0.y, fd0.y, iw.w0, iw.w1, ih.w0, ih.w1);
                const float y1 = bilerp_hw(fa1.y, fb1.y, fc1.y, fd1.y, iw.w0, iw.w1, ih.w0, ih.w1);
                o[q] = pack2(lerp_d(x0, x1, id.w0, id.w1), lerp_d(y0, y1, id.w0, id.w1), is_f16);
              }
            }
            const uint32_t dst = dst0 + (uint32_t)(r * 128) + (uint32_t)((c16 ^ (r & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3])
                         : "memory");
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("bar.sync 1, %0;" ::"n"(UP_THREADS) : "memory");
          if (tid == 0) mbar_arrive(plane_full(slot));
        }
        // hand back whatever is left of this chunk's low-resolution planes
        for (; released <= zl1; ++released) mbar_arrive(lp_empty((lseq_base + (unsigned)(released - zl0)) % LP_RING));
        lseq_base += (unsigned)(zl1 - zl0 + 1);
      }
    }
  } else if (warp < 4) {
    // ------------------------------- epilogue warps 0..3 -------------------------------
    const int row = warp * 32 + lane;
    const int lw = row & (SL_W - 1);
    const int lh = row >> 3;
    int buf = 0;
    uint32_t buf_phase = 0;
    for (int i = item_begin; i < item_end; ++i) {
      const SlabItem it = decode_item(p, item_at(i), Cfg::GROUP);
      const int oh = it.h0 + lh, ow = it.w0 + lw;
      // residual rows are loaded one 32-channel group ahead (also across the planes of the item); the first one
      // before the wait for the accumulator
      auto res_ptr = [&](int t) {
        const int od = it.q0 + t;
        const bool valid = (od < p.D) && (oh < p.H) && (ow < p.W);
        return residual_row(p.epi, valid, it.sample, od, oh, ow);
      };
      constexpr int GROUPS_PER_PLANE = BLOCK_N / 32;
      ResGroup res = load_residual_group(p.epi, res_ptr(0), 0);
      mbar_wait(tmem_full(buf), buf_phase);
      tcgen05_fence_after();
#pragma unroll 1
      for (int t = 0; t < SL_GROUP; ++t) {
        const int od = it.q0 + t;
        const bool valid = (od < p.D) && (oh < p.H) && (ow < p.W);
        const uint16_t *res_row = res_ptr(t);
        const uint32_t taddr = tmem_base + (uint32_t)((buf * SL_GROUP + t) * BLOCK_N) + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
        for (int gq = 0; gq < GROUPS_PER_PLANE; ++gq) {
          const int c0 = gq * 32;
          uint32_t v[32];
          tmem_ld_32x32b_x32(taddr + (uint32_t)c0, v);
          ResGroup next;
          if (gq + 1 < GROUPS_PER_PLANE) next = load_residual_group(p.epi, res_row, c0 + 32);
          else next = load_residual_group(p.epi, t + 1 < SL_GROUP ? res_ptr(t + 1) : nullptr, 0);
          tmem_wait_ld();
#ifndef DRAM_SLAB_EXPERIMENT_NO_EPILOGUE  // diagnostic builds only: results are wrong without it
          if (valid) epilogue_group<BLOCK_N == 32>(p.epi, v, c0, it.sample, od, oh, ow, res);
#endif
          res = next;
        }
      }
      tcgen05_fence_before();
      mbar_arrive(tmem_empty(buf));
      if (++buf == 2) {
        buf = 0;
        buf_phase ^= 1u;
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == SL_MMA_WARP) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------
// Streaming variant for Cin 64 -> Cout 32 (us3, med3d.py:90): the 27 taps (108 KiB) stay RESIDENT in shared memory,
// so nothing forces work items of a few planes.  The CTA walks a column plane by plane; input plane z feeds output
// planes z-1, z, z+1 through kd = 2, 1, 0, whose accumulators are adjacent 32-column blocks of a 16-block TMEM ring —
// EVERY interior MMA is the full kd stack (N = 96), against an average of N = 64 over the 6 planes of a 4-plane item,
// and a plane is fetched once instead of 6/4 times.  The issue rate is what bounds this layer (each tcgen05.mma costs
// ~34 clk + max(N/2, (128+N)/4), DESIGN.md section 3): 37 MMAs of ~90 clk per output plane instead of 54 of ~82.
//
// Work = contiguous ranges of (column, output plane) steps, D fastest; a CTA's range is cut into segments, one per
// column it touches: output planes [t0, t1) <- input planes max(t0-1, 0) .. min(t1, D-1).  Roles as above (warps 0-3
// epilogue, 4 planes, 5 MMA, 6 loads the weights once).
// ----------------------------------------------------------------------------------------
struct StreamCfg {
  static constexpr int RING_ = 5;                            // plane slots
  static constexpr int W_HW_BYTES = 3 * 32 * 128;            // [kd=2; kd=1; kd=0] of one (kh,kw): 96 rows x 64 channels
  static constexpr int W_BYTES = 9 * W_HW_BYTES;             // 110592
  static constexpr int TMEM_BLOCKS = 16, TMEM_COLS = 512;    // ring of 32-column accumulators
  static constexpr int SMEM_BYTES = 1024 + RING_ * PLANE_PITCH + W_BYTES + 512;
};

struct StreamSeg {
  int sample, w0, h0, t0, t1;
};
// The segment that starts at position `pos` of the CTA's range [.., pos_end): with a work list, the run of entries that
// continue the same column plane by plane.
__device__ __forceinline__ StreamSeg stream_segment(const SlabParams &p, int pos, int pos_end) {
  StreamSeg s;
  const int step = p.items ? __ldg(p.items + pos) : pos;
  const int col = step / p.D;
  s.t0 = step - col * p.D;
  if (p.items) {
    int len = 1;
    while (pos + len < pos_end && s.t0 + len < p.D && __ldg(p.items + pos + len) == step + len) ++len;
    s.t1 = s.t0 + len;
  } else {
    const int left = pos_end - pos;
    s.t1 = s.t0 + left < p.D ? s.t0 + left : p.D;
  }
  const int per_sample = p.cols_w * p.cols_h;
  s.sample = col / per_sample;
  const int r = col - s.sample * per_sample;
  const int ih = r / p.cols_w;
  s.w0 = (r - ih * p.cols_w) * SL_W;
  s.h0 = ih * SL_H;
  return s;
}

// K steps 1..35 of one input plane of the streaming kernel (step 0 is issued block by block by the caller).
// WRAP: the plane's accumulator blocks wrap around the TMEM ring, so every step is two instructions.
template <bool WRAP>
__device__ __forceinline__ void stream_issue_plane(uint32_t d1, uint32_t d2, uint64_t da_plane, uint64_t db1,
                                                   uint64_t db2, uint32_t id1, uint32_t id2) {
#pragma unroll
  for (int hw = 0; hw < 9; ++hw) {
    const int kh = hw / 3, kw = hw - 3 * kh;
    const uint32_t row_off16 = (uint32_t)((kh * PL_W + kw) * 128) >> 4;
    const uint32_t w_off16 = (uint32_t)(hw * StreamCfg::W_HW_BYTES) >> 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (hw == 0 && k == 0) continue;
      umma_bf16(d1, da_plane + (uint64_t)(row_off16 + 2 * k), db1 + (uint64_t)(w_off16 + 2 * k), id1, 1u);
      if (WRAP) umma_bf16(d2, da_plane + (uint64_t)(row_off16 + 2 * k), db2 + (uint64_t)(w_off16 + 2 * k), id2, 1u);
    }
  }
}

__global__ void __launch_bounds__(SL_THREADS, 1)
conv3d_stream32_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                       const __grid_constant__ SlabParams p) {
  constexpr int RING = StreamCfg::RING_;
  constexpr int NBLK = StreamCfg::TMEM_BLOCKS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = smem_base + RING * PLANE_PITCH;
  const uint32_t bar_base = w_base + StreamCfg::W_BYTES;
  auto plane_addr = [&](int s) { return smem_base + (uint32_t)s * PLANE_PITCH; };
  auto plane_full = [&](int s) { return bar_base + 8u * s; };
  auto plane_empty = [&](int s) { return bar_base + 8u * (RING + s); };
  const uint32_t w_full = bar_base + 8u * (2 * RING);
  auto tmem_full = [&](unsigned b) { return bar_base + 8u * (2 * RING + 1 + b); };
  auto tmem_empty = [&](unsigned b) { return bar_base + 8u * (2 * RING + 1 + NBLK + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * RING + 1 + 2 * NBLK);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < RING; ++s) {
      mbar_init(plane_full(s), 1);
      mbar_init(plane_empty(s), 1);
    }
    mbar_init(w_full, 1);
    for (int b = 0; b < NBLK; ++b) {
      mbar_init(tmem_full(b), 1);
      mbar_init(tmem_empty(b), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == SL_MMA_WARP) tmem_alloc(tmem_slot, StreamCfg::TMEM_COLS);
  if (warp == SL_A_WARP && lane == 0) prefetch_tensormap(&map_a);
  if (warp == SL_B_WARP && lane == 0) prefetch_tensormap(&map_w);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);

  // positions in the work list, if there is one (a step's output plane depends only on planes t-1, t, t+1 and the
  // order of their MMAs, not on where its segment starts)
  const int steps_total = p.items ? *p.count : p.steps_total;
  const int step_begin = (int)(((long long)blockIdx.x * steps_total) / gridDim.x);
  const int step_end = (int)(((long long)(blockIdx.x + 1) * steps_total) / gridDim.x);

  if (warp == SL_B_WARP) {
    if (lane == 0) {  // the whole filter, once: 27 boxes of 32 rows x 64 channels
      mbar_expect_tx(w_full, StreamCfg::W_BYTES);
      for (int hw = 0; hw < 9; ++hw)
        for (int blk = 0; blk < 3; ++blk)
          tma_load_2d(w_base + (uint32_t)(hw * StreamCfg::W_HW_BYTES + blk * 32 * 128), &map_w, w_full,
                      ((2 - blk) * 9 + hw) * SL_BLOCK_K, 0);
    }
    __syncwarp();
  } else if (warp == SL_A_WARP) {
    if (lane == 0) {
      unsigned pseq = 0;
      for (int step = step_begin; step < step_end;) {
        const StreamSeg sg = stream_segment(p, step, step_end);
        const int z_first = sg.t0 > 0 ? sg.t0 - 1 : 0, z_last = sg.t1 < p.D ? sg.t1 : p.D - 1;
        for (int z = z_first; z <= z_last; ++z, ++pseq) {
          const int slot = pseq % RING;
          mbar_wait(plane_empty(slot), ((pseq / RING) & 1u) ^ 1u);
          mbar_expect_tx(plane_full(slot), PLANE_BYTES);
          tma_load_5d(plane_addr(slot), &map_a, plane_full(slot), 0, sg.w0 - 1, sg.h0 - 1, z, sg.sample);
        }
        step += sg.t1 - sg.t0;
      }
    }
    __syncwarp();
  } else if (warp == SL_MMA_WARP) {
    const uint32_t idesc1 = make_idesc_16bit(128, 32, p.epi.is_f16), idesc2 = make_idesc_16bit(128, 64, p.epi.is_f16),
                   idesc3 = make_idesc_16bit(128, 96, p.epi.is_f16);
    auto idesc_of = [&](int n) { return n == 1 ? idesc1 : (n == 2 ? idesc2 : idesc3); };
    const uint64_t desc_a_const = make_sw128_desc_sbo(0u, PL_W * 128, 0);
    mbar_wait(w_full, 0u);
    tcgen05_fence_after();
    uint32_t wb = __shfl_sync(0xffffffffu, w_base, 0);
    const uint64_t db_base = make_sw128_desc(0u) | (uint64_t)((wb & 0x3FFFFu) >> 4);
    unsigned pseq = 0, oseq0 = 0;
    for (int step = step_begin; step < step_end;) {
      const StreamSeg sg = stream_segment(p, step, step_end);
      const int z_first = sg.t0 > 0 ? sg.t0 - 1 : 0, z_last = sg.t1 < p.D ? sg.t1 : p.D - 1;
      for (int z = z_first; z <= z_last; ++z, ++pseq) {
        // output planes this input plane feeds: t = z-1 (kd 2), z (kd 1), z+1 (kd 0), clipped to the segment
        const int lo = z - 1 > sg.t0 ? z - 1 : sg.t0, hi = z + 1 < sg.t1 - 1 ? z + 1 : sg.t1 - 1;
        const int nblk = hi - lo + 1;
        // accumulator blocks touched for the first time by this plane have to be drained by the epilogue
        for (int t = (z == z_first ? lo : z + 1); t <= hi; ++t) {
          const unsigned o = oseq0 + (unsigned)(t - sg.t0);
          mbar_wait(tmem_empty(o % NBLK), ((o / NBLK) & 1u) ^ 1u);
        }
        const int slot = pseq % RING;
        mbar_wait(plane_full(slot), (pseq / RING) & 1u);
        tcgen05_fence_after();
        uint32_t pa = plane_addr(slot);
        pa = __shfl_sync(0xffffffffu, pa, 0);
        const uint64_t da_plane = desc_a_const | (uint64_t)((pa & 0x3FFFFu) >> 4);
        const unsigned b_lo = (oseq0 + (unsigned)(lo - sg.t0)) % NBLK;
        const int n1 = nblk < (int)(NBLK - b_lo) ? nblk : (int)(NBLK - b_lo), n2 = nblk - n1;  // ring wrap: two runs
        const int bblk = lo - z + 1;  // weight block (0 = kd 2) of the first output plane
        const uint32_t d1 = tmem_base + b_lo * 32u, d2 = tmem_base;
        const uint64_t db1 = db_base + (uint64_t)((bblk * 32 * 128) >> 4), db2 = db1 + (uint64_t)((n1 * 32 * 128) >> 4);
        const uint32_t id1 = idesc_of(n1), id2 = idesc_of(n2 > 0 ? n2 : 1);
        const bool fresh_all = z == z_first;
        if (elect_one_sync()) {
          // (kh,kw) = (0,0), K step 0, block by block: a block's first MMA overwrites, the others accumulate
          for (int q = 0; q < nblk; ++q) {
            const int t = lo + q;
            const unsigned bq = (b_lo + (unsigned)q) % NBLK;
            umma_bf16(tmem_base + bq * 32u, da_plane, db1 + (uint64_t)((q * 32 * 128) >> 4), idesc1,
                      (fresh_all || t == z + 1) ? 0u : 1u);
          }
          // The other 35 K steps.  14 planes of 16 take the first branch: ONE instruction per step (two uniform 64-bit
          // adds each).  Keeping the ring-wrap instruction predicated in the same loop made the issuing thread the
          // bottleneck: predicated-off uniform instructions still wait on the scoreboard (ncu source view, round 2).
          if (n2 == 0) {
            stream_issue_plane<false>(d1, d2, da_plane, db1, db2, id1, id2);
          } else {
            stream_issue_plane<true>(d1, d2, da_plane, db1, db2, id1, id2);
          }
          umma_commit(plane_empty(slot));
          if (z - 1 >= sg.t0) umma_commit(tmem_full((oseq0 + (unsigned)(z - 1 - sg.t0)) % NBLK));
          if (z == p.D - 1 && sg.t1 == p.D) umma_commit(tmem_full((oseq0 + (unsigned)(z - sg.t0)) % NBLK));
        }
        __syncwarp();
      }
      oseq0 += (unsigned)(sg.t1 - sg.t0);
      step += sg.t1 - sg.t0;
    }
    __syncwarp();
  } else if (warp < 4) {
    const int row = warp * 32 + lane;
    const int lw = row & (SL_W - 1), lh = row >> 3;
    unsigned oseq = 0;
    for (int step = step_begin; step < step_end;) {
      const StreamSeg sg = stream_segment(p, step, step_end);
      const int oh = sg.h0 + lh, ow = sg.w0 + lw;
      const bool valid = oh < p.H && ow < p.W;
#pragma unroll 1
      for (int t = sg.t0; t < sg.t1; ++t, ++oseq) {
        const unsigned blk = oseq % NBLK;
        const ResGroup res = load_residual_group(p.epi, residual_row(p.epi, valid, sg.sample, t, oh, ow), 0);
        mbar_wait(tmem_full(blk), (oseq / NBLK) & 1u);
        tcgen05_fence_after();
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + blk * 32u + ((uint32_t)(warp * 32) << 16), v);
        tmem_wait_ld();
        tcgen05_fence_before();
        mbar_arrive(tmem_empty(blk));  // the block's values are in registers: hand it back before the arithmetic
        if (valid) epilogue_group<true>(p.epi, v, 0, sg.sample, t, oh, ow, res);
      }
      step += sg.t1 - sg.t0;
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == SL_MMA_WARP) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, StreamCfg::TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------
// host
// ----------------------------------------------------------------------------------------
int slab_plan_supported(const dram_conv_desc *d) {
  // Cout 128 (layer2 of the basic-block nets, the 3x3x3 of layer2's bottlenecks): two output planes per item; the
  // per-tap tile kernel pulls 32 KiB of operands per 392 MMA clocks through L2 there and reached 31 % tensor-pipe
  // utilisation (profiles/tensor_pipe_r2b.md).  DRAM_B200_SLAB128=0 keeps those layers on the tile kernel.
  const char *k128 = getenv("DRAM_B200_SLAB128");
  const bool allow128 = !(k128 && atoi(k128) == 0) && d->n_heads == 0;
  return d->kd == 3 && d->kh == 3 && d->kw == 3 && d->sd == 1 && d->sh == 1 && d->sw == 1 && d->dd == 1 &&
         d->dh == 1 && d->dw == 1 && d->pd == 1 && d->ph == 1 && d->pw == 1 &&
         (d->cout == 32 || d->cout == 64 || (d->cout == 128 && allow128));
}

template <int BN, bool UP>
static int slab_set_attr() {
  return check_cuda(cudaFuncSetAttribute(conv3d_slab_kernel<BN, UP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         SlabCfg<BN, UP>::SMEM_BYTES),
                    "cudaFuncSetAttribute(conv3d_slab_kernel)");
}

// ATen's align_corners source index on the host (same fp32 arithmetic as lin_index_ac).
static void host_lin_index(int dst, float scale, int in_size, int *i0, int *i1) {
  const float real = scale * (float)dst;
  int a = (int)real;
  if (a > in_size - 1) a = in_size - 1;
  *i0 = a;
  *i1 = a + ((a < in_size - 1) ? 1 : 0);
}
// Largest low-resolution extent read by any window of `win` consecutive outputs starting at k*step - 1.
static int max_src_span(int out_size, int in_size, int step, int win) {
  const float scale = ac_scale(in_size, out_size);
  int worst = 0;
  for (int o0 = -1; o0 < out_size; o0 += step) {
    int lo0, lo1, hi0, hi1;
    const int a = o0 < 0 ? 0 : o0, b = o0 + win - 1 > out_size - 1 ? out_size - 1 : o0 + win - 1;
    host_lin_index(a, scale, in_size, &lo0, &lo1);
    host_lin_index(b, scale, in_size, &hi0, &hi1);
    if (hi1 - lo0 + 1 > worst) worst = hi1 - lo0 + 1;
  }
  return worst;
}

int encode_act_map_plain(CUtensorMap *map, const void *base, int n, int d, int h, int w, int c, int box_c, int bw,
                         int bh, int is_f16);

int slab_plan_fill(dram_conv_plan *pl, const dram_conv_desc *d, const void *src1, const void *src2,
                   const void *weight, const EpiParams &epi) {
  pl->kind = 1;
  SlabParams &sp = pl->sp;
  sp.n = d->n; sp.D = d->di; sp.H = d->hi; sp.W = d->wi;
  sp.cols_w = ceil_div(d->wi, SL_W);
  sp.cols_h = ceil_div(d->hi, SL_H);
  const int group = slab_group(d->cout);
  sp.groups_d = ceil_div(d->di, group);
  const int64_t items = (int64_t)d->n * sp.cols_w * sp.cols_h * sp.groups_d;
  if (items > 0x7fffffffLL) {
    set_error("conv3d(planes): too many work items");
    return DRAM_E_ARG;
  }
  sp.items_total = (int)items;
  sp.chunks1 = d->c1 / SL_BLOCK_K;
  sp.chunks_total = (d->c1 + d->c2) / SL_BLOCK_K;
  const char *knob = getenv("DRAM_B200_DESC_BASE_OFFSET");
  sp.desc_base_offset_mode = knob ? atoi(knob) : 0;
  sp.up2x = d->src1_up2x ? 1 : 0;
  if (sp.up2x) {
    if (d->cout != 64 || d->c2 <= 0 || (d->di & 1) || (d->hi & 1) || (d->wi & 1)) {
      set_error("conv3d: src1_up2x needs cout == 64, a second source and even D, H, W (got cout %d, c2 %d, %dx%dx%d)",
                d->cout, d->c2, d->di, d->hi, d->wi);
      return DRAM_E_ARG;
    }
    sp.Dl = d->di / 2; sp.Hl = d->hi / 2; sp.Wl = d->wi / 2;
    sp.up_sd = ac_scale(sp.Dl, d->di); sp.up_sh = ac_scale(sp.Hl, d->hi); sp.up_sw = ac_scale(sp.Wl, d->wi);
    if (max_src_span(d->hi, sp.Hl, SL_H, PL_H) > LP_H || max_src_span(d->wi, sp.Wl, SL_W, PL_W) > LP_W) {
      set_error("conv3d: src1_up2x low-resolution patch exceeds %dx%d for %dx%d planes", LP_H, LP_W, d->hi, d->wi);
      return DRAM_E_ARG;
    }
  }
  sp.items = sp.count = nullptr;
  sp.epi = epi;
  // Cin 64 -> Cout 32 with one source (us3): weights-resident streaming kernel; DRAM_B200_US3=ring keeps the items
  const char *us3 = getenv("DRAM_B200_US3");
  sp.stream = (d->cout == 32 && sp.chunks_total == 1 && !sp.up2x && !(us3 && strcmp(us3, "ring") == 0)) ? 1 : 0;
  const int64_t steps = (int64_t)d->n * sp.cols_w * sp.cols_h * d->di;
  if (steps > 0x7fffffffLL) {
    set_error("conv3d(planes): too many plane steps");
    return DRAM_E_ARG;
  }
  sp.steps_total = (int)steps;
  pl->block_n = d->cout;
  pl->stages = sp.up2x ? RING_UP : RING;
  pl->m_tiles = sp.stream ? sp.steps_total : sp.items_total * group;
  pl->n_tiles = 1;
  const int64_t ktot = 27LL * (d->c1 + d->c2);
  int rc;
  if (sp.up2x)
    rc = encode_act_map_plain(&pl->map_a1, src1, d->n, sp.Dl, sp.Hl, sp.Wl, d->c1, SL_BLOCK_K, LP_W, LP_H, epi.is_f16);
  else
    rc = encode_act_map(&pl->map_a1, src1, d->n, d->di, d->hi, d->wi, d->c1, SL_BLOCK_K, PL_W, PL_H, 1, 1, 1, 1,
                        epi.is_f16);
  if (rc == DRAM_OK) {
    if (d->c2 > 0)
      rc = encode_act_map(&pl->map_a2, src2, d->n, d->di, d->hi, d->wi, d->c2, SL_BLOCK_K, PL_W, PL_H, 1, 1, 1, 1,
                          epi.is_f16);
    else
      pl->map_a2 = pl->map_a1;
  }
  if (rc == DRAM_OK) rc = encode_weight_map(&pl->map_w, weight, d->cout, ktot, d->cout, epi.is_f16);
  if (rc == DRAM_OK) {
    if (sp.up2x) {
      pl->smem_bytes = SlabCfg<64, true>::SMEM_BYTES;
      rc = slab_set_attr<64, true>();
    } else if (d->cout == 64) {
      pl->smem_bytes = SlabCfg<64>::SMEM_BYTES;
      rc = slab_set_attr<64, false>();
    } else if (d->cout == 128) {
      pl->smem_bytes = SlabCfg<128>::SMEM_BYTES;
      pl->stages = SlabCfg<128>::RING_;
      rc = slab_set_attr<128, false>();
    } else if (sp.stream) {
      pl->smem_bytes = StreamCfg::SMEM_BYTES;
      pl->stages = StreamCfg::RING_;
      rc = check_cuda(cudaFuncSetAttribute(conv3d_stream32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           StreamCfg::SMEM_BYTES),
                      "cudaFuncSetAttribute(conv3d_stream32_kernel)");
    } else {
      pl->smem_bytes = SlabCfg<32>::SMEM_BYTES;
      rc = slab_set_attr<32, false>();
    }
  }
  return rc;
}

int slab_plan_listable(const dram_conv_plan *pl) { return pl->sp.stream || (!pl->sp.up2x && pl->block_n == 64); }

// The work items of a listable plan: plane-ring items of 8 x 16 x 4 voxels or plane steps of 8 x 16 x 1 voxels, both
// numbered with D fastest.
int slab_plan_worklist(const dram_conv_plan *pl, const uint32_t *bits, int radius, uint8_t *flags, int *list, int *count,
                       cudaStream_t st) {
  const SlabParams &sp = pl->sp;
  return worklist_build(bits, sp.n, sp.D, sp.H, sp.W, SL_W, SL_H, sp.stream ? 1 : slab_group(pl->block_n), 1, radius,
                        flags, list, count, sp.stream ? sp.steps_total : sp.items_total, st);
}

int slab_plan_run(const dram_conv_plan *pl, int ctas, cudaStream_t st, const int *items, const int *count) {
  SlabParams sp = pl->sp;
  sp.items = items;
  sp.count = count;
  sp.epi = with_sat_counter(sp.epi);
  if (sp.stream) {
    if (sp.steps_total < ctas) ctas = sp.steps_total;
    conv3d_stream32_kernel<<<dim3(ctas), SL_THREADS, pl->smem_bytes, st>>>(pl->map_a1, pl->map_w, sp);
    DRAM_CHECK_LAUNCH("conv3d_stream32_kernel launch");
    return DRAM_OK;
  }
  if (pl->sp.items_total < ctas) ctas = pl->sp.items_total;
  dim3 grid(ctas);
  if (sp.up2x)
    conv3d_slab_kernel<64, true><<<grid, SlabCfg<64, true>::THREADS, pl->smem_bytes, st>>>(pl->map_a1, pl->map_a2,
                                                                                          pl->map_w, sp);
  else if (pl->block_n == 64)
    conv3d_slab_kernel<64, false><<<grid, SL_THREADS, pl->smem_bytes, st>>>(pl->map_a1, pl->map_a2, pl->map_w, sp);
  else if (pl->block_n == 128)
    conv3d_slab_kernel<128, false><<<grid, SL_THREADS, pl->smem_bytes, st>>>(pl->map_a1, pl->map_a2, pl->map_w, sp);
  else
    conv3d_slab_kernel<32, false><<<grid, SL_THREADS, pl->smem_bytes, st>>>(pl->map_a1, pl->map_a2, pl->map_w, sp);
  DRAM_CHECK_LAUNCH("conv3d_slab_kernel launch");
  return DRAM_OK;
}

}  // namespace dram
