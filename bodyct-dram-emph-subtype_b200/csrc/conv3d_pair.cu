// K1, M256 variant of the per-tap tile kernel for the wide layers (Cout a multiple of 256 with a long K loop:
// layer3 / layer4 of the basic-block nets, the 3x3x3 convolutions of the bottleneck nets' layer3 / layer4).
//
// Why: with a 128-voxel tile every (tap, chunk) stage moves a 16 KiB activation brick and a 32 KiB weight tile
// for 128 x 256 x 64 MACs — 48 KiB per 512 tensor-core clocks, ~56 % of the L2->SM peak on its own (ncu
// l1tex__m_xbar2l1tex_read_bytes, profiles/conv_ncu_r1f.md) with only four stages (2048 clocks) of look-ahead.
// Here one CTA computes a brick of 256 voxels, two 128-row boxes, against the same weight tile:
//   stage = [A box 0 | A box 1 | B] = 64 KiB for 2 x 128 x 256 x 64 MACs (1024 clocks): a third less
//   operand traffic per MAC and three stages = 3072 clocks of look-ahead;
//   accumulators: box 0 in TMEM columns [0,256), box 1 in [256,512) — all of TMEM, so the epilogue of a tile
//   is not overlapped with the next tile's MMAs; with K >= 108 chunks per tile that costs a few per cent;
//   epilogue: eight warps, warps 0-3 drain box 0 and warps 6-9 box 1 (TMEM lane quarter = warp % 4).
// The brick (p.bw x p.bh x p.bd voxels of p.bn samples) is split into its two boxes along the sample axis when it
// folds samples, else along one spatial axis.  A tap is skipped when the whole brick lies in the zero padding.
//
// Roles (320 threads): warps 0-3 / 6-9 epilogue, warp 4 lane 0 TMA producer, warp 5 MMA issuer (owns TMEM).
#include "conv_plan.h"

namespace dram {

static constexpr int P_BLOCK_N = 256;
static constexpr int P_BLOCK_K = 64;
static constexpr int P_A_BYTES = 128 * P_BLOCK_K * 2;          // one brick: 16 KiB
static constexpr int P_B_BYTES = P_BLOCK_N * P_BLOCK_K * 2;    // 32 KiB
static constexpr int P_STAGE_BYTES = 2 * P_A_BYTES + P_B_BYTES;  // 64 KiB
static constexpr int P_STAGES = 3;
static constexpr int P_THREADS = 320;
static constexpr int P_PRODUCER_WARP = 4, P_MMA_WARP = 5;
static constexpr int P_TMEM_COLS = 512;
static constexpr int P_SMEM_BYTES = 1024 + P_STAGES * P_STAGE_BYTES + 256;

// Origins of the two boxes of a brick: box 1 is box 0 moved by the half of the brick along its split axis.  A box
// past the end of the volume or batch is loaded out of bounds (zeros) and its rows are never stored.
struct PairCoord {
  TileCoord t[2];
};
__device__ __forceinline__ PairCoord decode_pair(const ConvKParams &p, int tile) {
  PairCoord pc;
  pc.t[0] = decode_tile(p, tile, P_BLOCK_N);
  pc.t[1] = pc.t[0];
  pc.t[1].w0 += p.bw - p.tw;  // the brick is twice the box along exactly one axis
  pc.t[1].h0 += p.bh - p.th;
  pc.t[1].d0 += p.bd - p.td;
  pc.t[1].sample += p.bn - p.tn;
  return pc;
}

__global__ void __launch_bounds__(P_THREADS, 1)
conv3d_pair_kernel(const __grid_constant__ CUtensorMap map_a1, const __grid_constant__ CUtensorMap map_a2,
                   const __grid_constant__ CUtensorMap map_w, const __grid_constant__ ConvKParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + P_STAGES * P_STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (P_STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * P_STAGES);
  const uint32_t tmem_empty_bar = bar_base + 8u * (2 * P_STAGES + 1);
  const uint32_t tmem_slot = bar_base + 8u * (2 * P_STAGES + 2);
  auto smem_a = [&](int s, int b) { return smem_base + (uint32_t)(s * P_STAGE_BYTES + b * P_A_BYTES); };
  auto smem_b = [&](int s) { return smem_base + (uint32_t)(s * P_STAGE_BYTES + 2 * P_A_BYTES); };

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < P_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(tmem_empty_bar, 256);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == P_MMA_WARP) tmem_alloc(tmem_slot, P_TMEM_COLS);
  if (warp == P_PRODUCER_WARP && lane == 0) {
    prefetch_tensormap(&map_a1);
    prefetch_tensormap(&map_a2);
    prefetch_tensormap(&map_w);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);

  if (warp == P_PRODUCER_WARP) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int i = blockIdx.x; i < p.total_tiles; i += gridDim.x) {
        const PairCoord pc = decode_pair(p, tile_at(p, i));
        for (int zd = 0; zd < p.kd; ++zd)
          for (int zh = 0; zh < p.kh; ++zh)
            for (int zw = 0; zw < p.kw; ++zw) {
              if (brick_tap_is_padding(p, pc.t[0], zd, zh, zw)) continue;
              const int tap = (zd * p.kh + zh) * p.kw + zw;
              for (int ch = 0; ch < p.chunks_total; ++ch) {
                mbar_wait(empty_bar(stage), phase ^ 1u);
                mbar_expect_tx(full_bar(stage), P_STAGE_BYTES);
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                  const TileCoord &t = pc.t[b];
                  const int iw0 = t.w0 * p.sw + zw * p.dw - p.pw, ih0 = t.h0 * p.sh + zh * p.dh - p.ph;
                  const int id0 = t.d0 * p.sd + zd * p.dd - p.pd;
                  if (ch < p.chunks1)
                    tma_load_5d(smem_a(stage, b), &map_a1, full_bar(stage), ch * P_BLOCK_K, iw0, ih0, id0, t.sample);
                  else
                    tma_load_5d(smem_a(stage, b), &map_a2, full_bar(stage), (ch - p.chunks1) * P_BLOCK_K, iw0, ih0,
                                id0, t.sample);
                }
                tma_load_2d(smem_b(stage), &map_w, full_bar(stage), (tap * p.chunks_total + ch) * P_BLOCK_K,
                            pc.t[0].n0);
                if (++stage == P_STAGES) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
            }
      }
    }
    __syncwarp();
  } else if (warp == P_MMA_WARP) {
    const uint32_t idesc = make_idesc_16bit(128, P_BLOCK_N, p.epi.is_f16);
    int stage = 0;
    uint32_t phase = 0, acc_phase = 0;
    for (int i = blockIdx.x; i < p.total_tiles; i += gridDim.x) {
      const PairCoord pc = decode_pair(p, tile_at(p, i));
      mbar_wait(tmem_empty_bar, acc_phase ^ 1u);  // the epilogue has drained both accumulators
      tcgen05_fence_after();
      uint32_t accumulate = 0;
      for (int zd = 0; zd < p.kd; ++zd)
        for (int zh = 0; zh < p.kh; ++zh)
          for (int zw = 0; zw < p.kw; ++zw) {
            if (brick_tap_is_padding(p, pc.t[0], zd, zh, zw)) continue;
            for (int ch = 0; ch < p.chunks_total; ++ch) {
              mbar_wait(full_bar(stage), phase);
              tcgen05_fence_after();
              const uint64_t da0 = make_sw128_desc(smem_a(stage, 0)), da1 = make_sw128_desc(smem_a(stage, 1));
              const uint64_t db = make_sw128_desc(smem_b(stage));
              if (elect_one_sync()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  umma_bf16(tmem_base, da0 + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (k > 0) ? 1u : accumulate);
                  umma_bf16(tmem_base + P_BLOCK_N, da1 + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc,
                            (k > 0) ? 1u : accumulate);
                }
                umma_commit(empty_bar(stage));
              }
              __syncwarp();
              accumulate = 1;
              if (++stage == P_STAGES) {
                stage = 0;
                phase ^= 1u;
              }
            }
          }
      if (elect_one_sync()) umma_commit(tmem_full_bar);
      __syncwarp();
      acc_phase ^= 1u;
    }
  } else {
    // ------------------------------- epilogue: warps 0-3 box 0, warps 6-9 box 1 -------------------------------
    const int quarter = warp & 3, brick = warp < 4 ? 0 : 1;
    const int row = quarter * 32 + lane;
    const int lw = row & (p.tw - 1);
    const int lh = (row >> p.tw_log2) & (p.th - 1);
    const int ld = (row >> (p.tw_log2 + p.th_log2)) & (p.td - 1);
    const int ls = row >> (p.tw_log2 + p.th_log2 + p.td_log2);
    uint32_t acc_phase = 0;
    for (int i = blockIdx.x; i < p.total_tiles; i += gridDim.x) {
      const PairCoord pc = decode_pair(p, tile_at(p, i));
      const TileCoord &t = pc.t[brick];
      const int od = t.d0 + ld, oh = t.h0 + lh, ow = t.w0 + lw, os = t.sample + ls;
      const bool valid = (os < p.n) && (od < p.Do) && (oh < p.Ho) && (ow < p.Wo);
      const uint16_t *res_row = residual_row(p.epi, valid, os, od, oh, ow);
      mbar_wait(tmem_full_bar, acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)(brick * P_BLOCK_N) + ((uint32_t)(quarter * 32) << 16);
      ResGroup res = load_residual_group(p.epi, res_row, t.n0);
#pragma unroll 1
      for (int c0 = 0; c0 < P_BLOCK_N; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + (uint32_t)c0, v);
        const ResGroup next = load_residual_group(p.epi, c0 + 32 < P_BLOCK_N ? res_row : nullptr, t.n0 + c0 + 32);
        tmem_wait_ld();
        if (valid) epilogue_group<false>(p.epi, v, t.n0 + c0, os, od, oh, ow, res);
        res = next;
      }
      tcgen05_fence_before();
      mbar_arrive(tmem_empty_bar);
      acc_phase ^= 1u;
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == P_MMA_WARP) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, P_TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------
// host (called from dram_conv3d_plan_create / dram_conv3d_run in conv3d_umma.cu)
// ----------------------------------------------------------------------------------------
int pair_plan_wanted(const dram_conv_desc *d, int block_n, int64_t k_chunks, int64_t pair_tiles) {
  // wide output, long K loop (the un-overlapped epilogue must stay a few per cent), no fused heads
  if (!(block_n == P_BLOCK_N && d->cout % P_BLOCK_N == 0 && k_chunks >= 64 && d->n_heads == 0 && d->store_out))
    return 0;
  const char *knob = getenv("DRAM_B200_PAIR_TILES");  // 0 = never, 1 = whenever possible, unset = heuristic
  if (knob) return atoi(knob) != 0;
  // Measured on B200 (DESIGN.md): +3 % on layer4 (512->512, 216 chunks) once the 256-voxel tiles fill >= 6 waves;
  // with fewer, larger tiles the last wave's idle SMs cost more than the saved operand traffic gains (layer3 at
  // batch 4: -12 %, everything at batch 1: -10 %).
  return k_chunks >= 200 && pair_tiles >= 6LL * sm_count();
}

int pair_plan_fill(dram_conv_plan *pl) {
  pl->pair = 1;
  pl->stages = P_STAGES;
  pl->smem_bytes = P_SMEM_BYTES;
  return check_cuda(cudaFuncSetAttribute(conv3d_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES),
                    "cudaFuncSetAttribute(conv3d_pair_kernel)");
}

int pair_plan_run(const dram_conv_plan *pl, int ctas, cudaStream_t st) {
  if (pl->p.total_tiles < ctas) ctas = pl->p.total_tiles;
  ConvKParams kp = pl->p;
  kp.epi = with_sat_counter(kp.epi);
  conv3d_pair_kernel<<<ctas, P_THREADS, pl->smem_bytes, st>>>(pl->map_a1, pl->map_a2, pl->map_w, kp);
  DRAM_CHECK_LAUNCH("conv3d_pair_kernel launch");
  return DRAM_OK;
}

}  // namespace dram
