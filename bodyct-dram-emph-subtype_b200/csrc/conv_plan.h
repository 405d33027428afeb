// The opaque plan behind dram_conv_plan: tensor maps + kernel parameters of either conv kernel.
#pragma once
#include "umma_common.cuh"

namespace dram {

// Per-tap TMA tile kernel (conv3d_umma.cu)
struct ConvKParams {
  int n, Do, Ho, Wo, Di, Hi, Wi;
  int tw, th, td, tn;          // A box = one 128-row MMA operand: tw x th x td voxels of tn samples (powers of two)
  int tw_log2, th_log2, td_log2;  // row -> (w,h,d,sample) decode: row = ((s*td + d)*th + h)*tw + w
  int bw, bh, bd, bn;          // brick = work unit of one tile: the box (M128 kernel) or two boxes (pair kernel)
  int tiles_w, tiles_h, tiles_d, tiles_per_sample, sample_groups, num_n_tiles, total_tiles;  // bricks along each axis
  int kd, kh, kw, sd, sh, sw, dd, dh, dw, pd, ph, pw;
  int chunks1, chunks_total;   // 64-channel chunks of source 1 / of both sources
  int staged_res;              // staged epilogue: 1 = the residual tile comes through TMA as well
  const int *order;            // tile walk order (descending executed stages), or null = tiles in index order
  EpiParams epi;
};


#ifdef __CUDACC__
struct TileCoord {
  int n0, sample, d0, h0, w0;
};
// Origin of the brick of tile index `tile` (n-tile fastest, then w, h, d, sample group); sample = its first sample.
__device__ __forceinline__ TileCoord decode_tile(const ConvKParams &p, int tile, int block_n) {
  TileCoord t;
  int n_tile = tile % p.num_n_tiles;
  int m_tile = tile / p.num_n_tiles;
  t.n0 = n_tile * block_n;
  const int group = m_tile / p.tiles_per_sample;
  int r = m_tile - group * p.tiles_per_sample;
  int iw = r % p.tiles_w;
  int r2 = r / p.tiles_w;
  int ih = r2 % p.tiles_h;
  int id = r2 / p.tiles_h;
  t.sample = group * p.bn;
  t.w0 = iw * p.bw;
  t.h0 = ih * p.bh;
  t.d0 = id * p.bd;
  return t;
}
// The i-th tile a persistent CTA works on: the plan's cost-sorted permutation when it has one.
__device__ __forceinline__ int tile_at(const ConvKParams &p, int i) { return p.order ? __ldg(p.order + i) : i; }

// True when every input coordinate the tile reads along one axis for this tap is padding.
__device__ __forceinline__ bool tap_is_padding(int i0, int extent, int stride, int in_size) {
  return (i0 + (extent - 1) * stride < 0) || (i0 >= in_size);
}
// True when the whole brick reads zero padding for this tap; every sample of the brick alike.
__device__ __forceinline__ bool brick_tap_is_padding(const ConvKParams &p, const TileCoord &t, int zd, int zh, int zw) {
  return tap_is_padding(t.d0 * p.sd + zd * p.dd - p.pd, p.bd, p.sd, p.Di) ||
         tap_is_padding(t.h0 * p.sh + zh * p.dh - p.ph, p.bh, p.sh, p.Hi) ||
         tap_is_padding(t.w0 * p.sw + zw * p.dw - p.pw, p.bw, p.sw, p.Wi);
}
#endif

// Plane-ring kernel (conv3d_slab.cu): 3x3x3, stride 1, dilation 1, Cout in {32, 64}
struct SlabParams {
  int n, D, H, W;              // input == output spatial dims
  int cols_w, cols_h, groups_d, items_total;
  int chunks1, chunks_total;
  int desc_base_offset_mode;   // experiment knob for the UMMA descriptor base-offset field (0 = leave 0)
  // source 1 given at half resolution and up-sampled x2 (trilinear, align_corners=True) by the kernel
  int up2x;                    // 0 / 1
  int Dl, Hl, Wl;              // low-resolution dims (D/2, H/2, W/2)
  float up_sd, up_sh, up_sw;   // ATen source scales (Dl-1)/(D-1) ...
  // weights-resident streaming kernel (Cin 64 -> Cout 32): work = (column, output plane) steps
  int stream;                  // 0 / 1
  int steps_total;             // n * cols_w * cols_h * D
  // optional work list (dram_conv3d_run_listed): the kernel runs items / steps items[0 .. *count) instead of all of
  // them; null = every item
  const int *items, *count;
  EpiParams epi;
};

}  // namespace dram

struct dram_conv_plan {
  int kind;  // 0 = per-tap tiles, 1 = plane ring
  CUtensorMap map_a1, map_a2, map_w;
  CUtensorMap map_out, map_res;  // staged (TMA store) epilogue of the tile kernel
  int staged;
  int pair;                      // 1 = M256 kernel (conv3d_pair.cu): two boxes share every weight tile
  int order_entries;             // entries of the tile order dram_conv3d_plan_set_order writes (0: no order needed)
  dram::ConvKParams p;
  dram::SlabParams sp;
  int block_n;
  int stages;
  size_t smem_bytes;
  int64_t flops;
  int m_tiles, n_tiles;
};
