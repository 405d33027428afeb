// Work lists that restrict the full-resolution decoder stage to the voxels the dRAM reads.
//
// predict_step uses the dense head maps (decoder grid d x h x w, the stem's output size) only through K7:
//   dRAM(D x H x W) = trilinear_align_corners(dense) x ess,
// which reads dense at the corners {i0, i1} per axis of every ess voxel (lin_index_ac; i1 is read even where its
// weight is 0).  Call that set R0.  A 3x3x3 convolution computes its output on R0 from its input on R0 (+) 1 (the box
// dilation by one voxel), so us3 + heads needs R0, us2.1 R0 (+) 1, us2.0 R0 (+) 2 and the K4 that feeds us2.0 R0 (+) 3.
// A work item (tile, slab item or plane step) of one of those kernels runs if its output box meets the layer's region;
// everything else keeps whatever the buffer held (zeros from the engine's construction, or finite activations of an
// earlier run), which no active item passes on to R0.
//
//   dram_decoder_support       ess -> R0 as a bit mask [n][d][h][words of w]   (two passes, x first, then y and z)
//   worklist_build             R0 -> active flags of a kernel's items -> compacted ascending list + count
// All integer work: the lists are the same for the same ess whatever the launch configuration.
#include "common.h"

namespace dram {

// Smallest source index x whose i0 can reach c (or 0): i0 is non-decreasing in x.
__device__ __forceinline__ int first_source(int c, float scale, int out_size, int in_size) {
  if (c <= 0 || scale <= 0.0f) return 0;
  int x = (int)((float)c / scale);
  if (x > out_size - 1) x = out_size - 1;
  while (x > 0 && lin_index_ac(x - 1, scale, in_size).i0 >= c) --x;
  return x;
}

// Pass 1: one thread per (sample, Z, Y, 32-column word of the decoder grid): bit j = some ess voxel of the row has
// c0 + j in {i0(x), i1(x)}.
__global__ void __launch_bounds__(256)
support_rows_kernel(const uint8_t *__restrict__ ess, uint32_t *__restrict__ rows, int64_t total, int W, int w,
                    int words, float sw) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(t % words);
    const uint8_t *e = ess + (t / words) * W;
    const int c0 = k * 32;
    uint32_t bits = 0;
    for (int x = first_source(c0 - 1, sw, W, w); x < W; ++x) {
      const LinIdx ix = lin_index_ac(x, sw, w);
      if (ix.i0 > c0 + 31) break;
      if (e[x]) {
        if (ix.i0 >= c0) bits |= 1u << (ix.i0 - c0);
        if (ix.i1 >= c0 && ix.i1 <= c0 + 31) bits |= 1u << (ix.i1 - c0);
      }
    }
    rows[t] = bits;
  }
}

// Pass 2: one thread per (sample, z, y, word) of R0: OR of the pass-1 rows (Z, Y) whose corners include (z, y).
__global__ void __launch_bounds__(256)
support_planes_kernel(const uint32_t *__restrict__ rows, uint32_t *__restrict__ bits, int n, int D, int H, int d,
                      int h, int words, float sd, float sh) {
  const int64_t total = (int64_t)n * d * h * words;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(t % words);
    int64_t r = t / words;
    const int y = (int)(r % h);
    r /= h;
    const int z = (int)(r % d);
    const int s = (int)(r / d);
    uint32_t acc = 0;
    for (int Z = first_source(z - 1, sd, D, d); Z < D; ++Z) {
      const LinIdx iz = lin_index_ac(Z, sd, d);
      if (iz.i0 > z) break;
      if (iz.i0 != z && iz.i1 != z) continue;
      for (int Y = first_source(y - 1, sh, H, h); Y < H; ++Y) {
        const LinIdx iy = lin_index_ac(Y, sh, h);
        if (iy.i0 > y) break;
        if (iy.i0 == y || iy.i1 == y) acc |= rows[(((int64_t)s * D + Z) * H + Y) * words + k];
      }
    }
    bits[t] = acc;
  }
}

// Item geometry of a kernel that takes a work list: output boxes of tw x th x td voxels, numbered with D fastest
// ((sample, h, w) column, then the group along D: plane-ring items and plane steps) or with W fastest (K4 tiles).
__global__ void __launch_bounds__(256)
worklist_flags_kernel(const uint32_t *__restrict__ bits, uint8_t *__restrict__ flags, int total, int d, int h, int w,
                      int words, int tw, int th, int td, int d_fastest, int radius) {
  const int tiles_w = (w + tw - 1) / tw, tiles_h = (h + th - 1) / th, tiles_d = (d + td - 1) / td;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int r = i, iw, ih, id;
    if (d_fastest) {
      id = r % tiles_d; r /= tiles_d;
      iw = r % tiles_w; r /= tiles_w;
      ih = r % tiles_h; r /= tiles_h;
    } else {
      iw = r % tiles_w; r /= tiles_w;
      ih = r % tiles_h; r /= tiles_h;
      id = r % tiles_d; r /= tiles_d;
    }
    const int s = r;
    const int z0 = max(id * td - radius, 0), z1 = min(id * td + td - 1 + radius, d - 1);
    const int y0 = max(ih * th - radius, 0), y1 = min(ih * th + th - 1 + radius, h - 1);
    const int x0 = max(iw * tw - radius, 0), x1 = min(iw * tw + tw - 1 + radius, w - 1);
    const int k0 = x0 >> 5, k1 = x1 >> 5;
    bool on = false;
    for (int z = z0; z <= z1 && !on; ++z)
      for (int y = y0; y <= y1 && !on; ++y) {
        const uint32_t *row = bits + (((int64_t)s * d + z) * h + y) * words;
        for (int k = k0; k <= k1; ++k) {
          uint32_t m = 0xffffffffu;
          if (k == k0) m &= 0xffffffffu << (x0 & 31);
          if (k == k1) m &= 0xffffffffu >> (31 - (x1 & 31));
          if (row[k] & m) {
            on = true;
            break;
          }
        }
      }
    flags[i] = on ? 1 : 0;
  }
}

// One CTA: the ascending indices of the set flags, and their number.  16 flags per thread and pass.
static constexpr int WL_THREADS = 1024, WL_PER_THREAD = 16;
__global__ void __launch_bounds__(WL_THREADS)
worklist_compact_kernel(const uint8_t *__restrict__ flags, int total, int *__restrict__ list, int *__restrict__ count) {
  __shared__ int warp_sum[WL_THREADS / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int base = 0;
  for (int start = 0; start < total; start += WL_THREADS * WL_PER_THREAD) {
    const int i0 = start + threadIdx.x * WL_PER_THREAD;
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < WL_PER_THREAD; ++j)
      if (i0 + j < total && flags[i0 + j]) m |= 1u << j;
    const int cnt = __popc(m);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sum[wid] = incl;
    __syncthreads();
    int before = 0, all = 0;
    for (int q = 0; q < WL_THREADS / 32; ++q) {
      const int v = warp_sum[q];
      if (q < wid) before += v;
      all += v;
    }
    int pos = base + before + incl - cnt;
    for (; m; m &= m - 1) list[pos++] = i0 + __ffs(m) - 1;
    base += all;
    __syncthreads();  // warp_sum is rewritten by the next pass
  }
  if (threadIdx.x == 0) *count = base;
}

int worklist_build(const uint32_t *bits, int n, int d, int h, int w, int tw, int th, int td, int d_fastest, int radius,
                   uint8_t *flags, int *list, int *count, int total, cudaStream_t st) {
  if (!bits || !flags || !list || !count || n <= 0 || d <= 0 || h <= 0 || w <= 0 || total <= 0 || radius < 0) {
    set_error("worklist: null buffer, empty grid or negative radius");
    return DRAM_E_ARG;
  }
  const int words = ceil_div(w, 32);
  worklist_flags_kernel<<<ceil_div(total, 256) < 4096 ? ceil_div(total, 256) : 4096, 256, 0, st>>>(
      bits, flags, total, d, h, w, words, tw, th, td, d_fastest, radius);
  DRAM_CHECK_LAUNCH("worklist_flags_kernel launch");
  worklist_compact_kernel<<<1, WL_THREADS, 0, st>>>(flags, total, list, count);
  DRAM_CHECK_LAUNCH("worklist_compact_kernel launch");
  return DRAM_OK;
}

}  // namespace dram

using namespace dram;

extern "C" int dram_decoder_support(const uint8_t *ess, int32_t n, int32_t D, int32_t H, int32_t W, int32_t d,
                                    int32_t h, int32_t w, uint32_t *rows, uint32_t *bits, void *stream) {
  DRAM_REQUIRE(ess && rows && bits, "dram_decoder_support: null pointer");
  DRAM_REQUIRE(n > 0 && D > 0 && H > 0 && W > 0 && d > 0 && h > 0 && w > 0 && d <= D && h <= H && w <= W,
               "dram_decoder_support: bad sizes (%d x %d x %d -> %d x %d x %d)", D, H, W, d, h, w);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int words = ceil_div(w, 32);
  const int64_t total_rows = (int64_t)n * D * H * words, total_bits = (int64_t)n * d * h * words;
  const int grid_rows = (int)(ceil_div64(total_rows, 256) < 8192 ? ceil_div64(total_rows, 256) : 8192);
  const int grid_bits = (int)(ceil_div64(total_bits, 256) < 8192 ? ceil_div64(total_bits, 256) : 8192);
  support_rows_kernel<<<grid_rows, 256, 0, st>>>(ess, rows, total_rows, W, w, words, ac_scale(w, W));
  DRAM_CHECK_LAUNCH("support_rows_kernel launch");
  support_planes_kernel<<<grid_bits, 256, 0, st>>>(rows, bits, n, D, H, d, h, words, ac_scale(d, D), ac_scale(h, H));
  DRAM_CHECK_LAUNCH("support_planes_kernel launch");
  return DRAM_OK;
}
