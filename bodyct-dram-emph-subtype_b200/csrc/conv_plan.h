// The opaque plan behind dram_conv_plan: tensor maps + kernel parameters of either conv kernel.
#pragma once
#include "umma_common.cuh"

namespace dram {

// Per-tap TMA tile kernel (conv3d_umma.cu)
struct ConvKParams {
  int n, Do, Ho, Wo, Di, Hi, Wi;
  int tw, th, td;              // tile extents (powers of two, product 128)
  int tw_log2, th_log2;        // row -> (w,h,d) decode
  int tiles_w, tiles_h, tiles_d, tiles_per_sample, num_n_tiles, total_tiles;
  int kd, kh, kw, sd, sh, sw, dd, dh, dw, pd, ph, pw;
  int chunks1, chunks_total;   // 64-channel chunks of source 1 / of both sources
  int staged_res;              // staged epilogue: 1 = the residual tile comes through TMA as well
  int m_tiles_total;           // pair kernel: number of 128-voxel bricks (tiles_per_sample * n)
  EpiParams epi;
};


#ifdef __CUDACC__
struct TileCoord {
  int n0, sample, d0, h0, w0;
};
__device__ __forceinline__ TileCoord decode_tile(const ConvKParams &p, int tile, int block_n) {
  TileCoord t;
  int n_tile = tile % p.num_n_tiles;
  int m_tile = tile / p.num_n_tiles;
  t.n0 = n_tile * block_n;
  t.sample = m_tile / p.tiles_per_sample;
  int r = m_tile - t.sample * p.tiles_per_sample;
  int iw = r % p.tiles_w;
  int r2 = r / p.tiles_w;
  int ih = r2 % p.tiles_h;
  int id = r2 / p.tiles_h;
  t.w0 = iw * p.tw;
  t.h0 = ih * p.th;
  t.d0 = id * p.td;
  return t;
}
// True when every input coordinate the tile reads along one axis for this tap is padding.
__device__ __forceinline__ bool tap_is_padding(int i0, int extent, int stride, int in_size) {
  return (i0 + (extent - 1) * stride < 0) || (i0 >= in_size);
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
  int pair;                      // 1 = M256 kernel (conv3d_pair.cu): two bricks share every weight tile
  dram::ConvKParams p;
  dram::SlabParams sp;
  int block_n;
  int stages;
  size_t smem_bytes;
  int64_t flops;
  int m_tiles, n_tiles;
};
