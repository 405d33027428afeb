// Device versions of the CPU steps either side of the network (SURVEY §8f rows f1, f2).
//
// f1  dataset.py:66-80  lung = lobe > 0; 2 x binary_dilation with the full 3x3x3 structure (== a 5x5x5 box
//                       maximum with a zero border); scan[outside] = -2048; bounding box of the lung grown by
//                       ceil(5 mm / spacing) (utils.py:53-63, the growth is applied by the caller); crop;
//                       ess = (scan < -910) & lung.  All integer/byte work: bit-exact.
// f2  processor.py:111-158 + utils.py:28-37  trilinear (align_corners=True) resample of a dRAM to the crop
//                       size, paste into the zero-filled full volume, clip to [0,1], x255 in fp64, truncate
//                       to uint8 — one pass over the output volume, only uint8 leaves the GPU.
#include <math.h>

#include <atomic>

#include "common.h"

namespace dram {

// ---------------------------------------------------------------------------------------
// bounding box of mask != 0: bbox = {zmin, zmax+1, ymin, ymax+1, xmin, xmax+1}; one warp per (z, y) row
// ---------------------------------------------------------------------------------------
__global__ void bbox_init_kernel(int *bbox, int D, int H, int W) {
  bbox[0] = D; bbox[1] = 0; bbox[2] = H; bbox[3] = 0; bbox[4] = W; bbox[5] = 0;
}
__global__ void __launch_bounds__(256)
mask_bbox_kernel(const uint8_t *__restrict__ mask, int *__restrict__ bbox, int D, int H, int W) {
  const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  const int rows = D * H;
  int zlo = D, zhi = 0, ylo = H, yhi = 0, xlo = W, xhi = 0;
  for (int r = blockIdx.x * warps + (threadIdx.x >> 5); r < rows; r += gridDim.x * warps) {
    const uint8_t *row = mask + (int64_t)r * W;
    int lo = W, hi = 0;
    for (int x = lane; x < W; x += 32)
      if (row[x]) {
        lo = min(lo, x);
        hi = max(hi, x + 1);
      }
    if (hi > 0) {
      const int z = r / H, y = r - z * H;
      xlo = min(xlo, lo); xhi = max(xhi, hi);
      zlo = min(zlo, z); zhi = max(zhi, z + 1);
      ylo = min(ylo, y); yhi = max(yhi, y + 1);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    zlo = min(zlo, __shfl_xor_sync(0xffffffffu, zlo, o)); zhi = max(zhi, __shfl_xor_sync(0xffffffffu, zhi, o));
    ylo = min(ylo, __shfl_xor_sync(0xffffffffu, ylo, o)); yhi = max(yhi, __shfl_xor_sync(0xffffffffu, yhi, o));
    xlo = min(xlo, __shfl_xor_sync(0xffffffffu, xlo, o)); xhi = max(xhi, __shfl_xor_sync(0xffffffffu, xhi, o));
  }
  if (lane == 0 && zhi > 0) {
    atomicMin(&bbox[0], zlo); atomicMax(&bbox[1], zhi);
    atomicMin(&bbox[2], ylo); atomicMax(&bbox[3], yhi);
    atomicMin(&bbox[4], xlo); atomicMax(&bbox[5], xhi);
  }
}

// ---------------------------------------------------------------------------------------
// f1 on bit masks.  The window is the crop grown by 2 voxels on every side (the reach of two dilations):
// bit (zz, yy, xx) of the window = voxel (z0 - 2 + zz, y0 - 2 + yy, x0 - 2 + xx), zero outside the volume.
//   pass A  lung_pack_bits_kernel      lobe > 0 -> one bit per voxel (a warp ballots 32 voxels of a row)
//   pass B  lung_dilate_bits_kernel    in-plane 5x5 maximum on 32-voxel words (shifts + the neighbour words' carry)
//   pass C  lung_crop_kernel           5-plane maximum of pass B + blanking + crop + masks, 8 voxels per thread,
//                                      16- and 8-byte stores
// Round 1 did the same arithmetic one byte at a time (25 byte loads and two 64-bit divisions per voxel, byte stores):
// 0.40 ms per 256^3 volume against ~0.03 ms of compulsory traffic.
// ---------------------------------------------------------------------------------------
struct BitWindow {
  int wd, wh, ww;  // planes, rows, 32-bit words per row of the window
};
__host__ __device__ inline BitWindow bit_window(int cd, int ch, int cw) {
  BitWindow b;
  b.wd = cd + 4;
  b.wh = ch + 4;
  b.ww = (cw + 4 + 31) / 32;
  return b;
}

__global__ void __launch_bounds__(256)
lung_pack_bits_kernel(const uint8_t *__restrict__ lobe, uint32_t *__restrict__ bits, int D, int H, int W, int z0, int y0,
                      int x0, int cd, int ch, int cw) {
  const BitWindow bw = bit_window(cd, ch, cw);
  const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  const int rows = bw.wd * bw.wh;
  for (int r = blockIdx.x * warps + (threadIdx.x >> 5); r < rows; r += gridDim.x * warps) {
    const int zz = r / bw.wh, yy = r - zz * bw.wh;
    const int gz = z0 - 2 + zz, gy = y0 - 2 + yy;
    const bool row_ok = gz >= 0 && gz < D && gy >= 0 && gy < H;
    const uint8_t *row = lobe + ((int64_t)(row_ok ? gz : 0) * H + (row_ok ? gy : 0)) * W;
    uint32_t *orow = bits + (int64_t)r * bw.ww;
    for (int w = 0; w < bw.ww; ++w) {
      const int gx = x0 - 2 + w * 32 + lane;
      const bool on = row_ok && gx >= 0 && gx < W && row[gx] != 0;
      const uint32_t word = __ballot_sync(0xffffffffu, on);
      if (lane == 0) orow[w] = word;
    }
  }
}

// 5-wide maximum along x of a row of bit words: bit i of the result = OR of bits i-2 .. i+2.
__device__ __forceinline__ uint32_t xdil5(uint32_t left, uint32_t mid, uint32_t right) {
  return mid | (mid << 1) | (mid << 2) | (mid >> 1) | (mid >> 2) | (left >> 31) | (left >> 30) | (right << 31) |
         (right << 30);
}
__global__ void __launch_bounds__(256)
lung_dilate_bits_kernel(const uint32_t *__restrict__ bits, uint32_t *__restrict__ out, int cd, int ch, int cw) {
  const BitWindow bw = bit_window(cd, ch, cw);
  const int64_t total = (int64_t)bw.wd * bw.wh * bw.ww;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(t % bw.ww);
    const int64_t r = t / bw.ww;
    const int yy = (int)(r % bw.wh);
    const uint32_t *plane = bits + (r - yy) * bw.ww;
    uint32_t acc = 0;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
      const int y2 = yy + dy;
      if (y2 < 0 || y2 >= bw.wh) continue;
      const uint32_t *row = plane + (int64_t)y2 * bw.ww;
      acc |= xdil5(w > 0 ? row[w - 1] : 0u, row[w], w + 1 < bw.ww ? row[w + 1] : 0u);
    }
    out[t] = acc;
  }
}

// Pass C.  The crop is one flat array of cd*ch*cw voxels; a thread owns 8 consecutive ones (a 16-byte store of the
// image, 8-byte stores of the masks; a group may run over a row end).  Voxels past the end are handled by the last
// thread one by one.
__global__ void __launch_bounds__(256)
lung_crop_kernel(const short *__restrict__ scan, const uint8_t *__restrict__ lobe, const uint32_t *__restrict__ dil,
                 short *__restrict__ image_c, uint8_t *__restrict__ lung_c, uint8_t *__restrict__ ess_c, int D, int H,
                 int W, int z0, int y0, int x0, int cd, int ch, int cw, short blank, short ess_below, int vec_ok) {
  const BitWindow bw = bit_window(cd, ch, cw);
  const int64_t total = (int64_t)cd * ch * cw;
  const int64_t groups = (total + 7) / 8;
  const int64_t wplane = (int64_t)bw.wh * bw.ww;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t0 = g * 8;
    int x = (int)(t0 % cw);
    const int64_t r = t0 / cw;
    int y = (int)(r % ch);
    int z = (int)(r / ch);
    short v8[8];
    uint8_t l8[8], e8[8];
    int word_idx = -1, word_y = -1, word_z = -1;
    uint32_t word = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v8[j] = 0; l8[j] = 0; e8[j] = 0;
      if (t0 + j < total) {
        const int bx = x + 2, wi = bx >> 5;
        if (wi != word_idx || y != word_y || z != word_z) {  // twice-dilated lung: OR of window planes z .. z+4
          const uint32_t *p = dil + (int64_t)z * wplane + (int64_t)(y + 2) * bw.ww + wi;
          word = p[0] | p[wplane] | p[2 * wplane] | p[3 * wplane] | p[4 * wplane];
          word_idx = wi; word_y = y; word_z = z;
        }
        const int64_t src = ((int64_t)(z0 + z) * H + (y0 + y)) * W + (x0 + x);
        const short v = ((word >> (bx & 31)) & 1u) ? scan[src] : blank;
        const uint8_t lung = lobe[src] ? 1 : 0;
        v8[j] = v; l8[j] = lung; e8[j] = (v < ess_below && lung) ? 1 : 0;
        if (++x == cw) {
          x = 0;
          if (++y == ch) { y = 0; ++z; }
        }
      }
    }
    if (vec_ok && t0 + 8 <= total) {
      uint4 vi;
      vi.x = (uint32_t)(uint16_t)v8[0] | ((uint32_t)(uint16_t)v8[1] << 16);
      vi.y = (uint32_t)(uint16_t)v8[2] | ((uint32_t)(uint16_t)v8[3] << 16);
      vi.z = (uint32_t)(uint16_t)v8[4] | ((uint32_t)(uint16_t)v8[5] << 16);
      vi.w = (uint32_t)(uint16_t)v8[6] | ((uint32_t)(uint16_t)v8[7] << 16);
      *reinterpret_cast<uint4 *>(image_c + t0) = vi;
      uint2 vl, ve;
      vl.x = l8[0] | (l8[1] << 8) | (l8[2] << 16) | ((uint32_t)l8[3] << 24);
      vl.y = l8[4] | (l8[5] << 8) | (l8[6] << 16) | ((uint32_t)l8[7] << 24);
      ve.x = e8[0] | (e8[1] << 8) | (e8[2] << 16) | ((uint32_t)e8[3] << 24);
      ve.y = e8[4] | (e8[5] << 8) | (e8[6] << 16) | ((uint32_t)e8[7] << 24);
      *reinterpret_cast<uint2 *>(lung_c + t0) = vl;
      *reinterpret_cast<uint2 *>(ess_c + t0) = ve;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (t0 + j < total) {
          image_c[t0 + j] = v8[j];
          lung_c[t0 + j] = l8[j];
          ess_c[t0 + j] = e8[j];
        }
    }
  }
}

// ---------------------------------------------------------------------------------------
// f2: full-volume uint8 heat-map from one network-size dRAM.
// ---------------------------------------------------------------------------------------
// One warp per output row.  The x interpolation (index pair + weights) is the same for every row: a table in shared
// memory, built once per CTA.  A dRAM is zero outside `ess` (~2 % of a chest volume), so most 32-voxel stretches read
// eight zeros: those skip the arithmetic (0 -> 0 exactly).
struct XEntry {
  int i0, i1;
  float w0, w1;
};
__global__ void __launch_bounds__(256)
heatmap_u8_kernel(const float *__restrict__ map, uint8_t *__restrict__ out, int d, int h, int w, int OD, int OH,
                  int OW, int z0, int y0, int x0, int cd, int ch, int cw, float sd, float sh, float sw) {
  extern __shared__ XEntry xtab[];  // cw entries
  for (int x = threadIdx.x; x < cw; x += blockDim.x) {
    const LinIdx iw = lin_index_ac(x, sw, w);
    xtab[x] = XEntry{iw.i0, iw.i1, iw.w0, iw.w1};
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  const int rows = OD * OH;
  for (int r = blockIdx.x * warps + (threadIdx.x >> 5); r < rows; r += gridDim.x * warps) {
    const int gz = r / OH, gy = r - gz * OH;
    uint8_t *orow = out + (int64_t)r * OW;
    const int z = gz - z0, y = gy - y0;
    if (z < 0 || z >= cd || y < 0 || y >= ch) {
      for (int x = lane; x < OW; x += 32) orow[x] = 0;
      continue;
    }
    const LinIdx id = lin_index_ac(z, sd, d), ih = lin_index_ac(y, sh, h);
    const float *r00 = map + ((int64_t)id.i0 * h + ih.i0) * w, *r01 = map + ((int64_t)id.i0 * h + ih.i1) * w;
    const float *r10 = map + ((int64_t)id.i1 * h + ih.i0) * w, *r11 = map + ((int64_t)id.i1 * h + ih.i1) * w;
    // four 32-voxel stretches per trip: their 32 loads are issued before any of them is used
    for (int gx0 = 0; gx0 < OW; gx0 += 128) {
      float a0[4], a1[4], b0[4], b1[4], c0[4], c1[4], e0[4], e1[4];
      XEntry xe[4];
      bool in[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int gx = gx0 + 32 * q + lane, x = gx - x0;
        in[q] = gx < OW && x >= 0 && x < cw;
        xe[q] = in[q] ? xtab[x] : XEntry{0, 0, 0.f, 0.f};
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        a0[q] = a1[q] = b0[q] = b1[q] = c0[q] = c1[q] = e0[q] = e1[q] = 0.f;
        if (in[q]) {
          a0[q] = __ldg(r00 + xe[q].i0); a1[q] = __ldg(r00 + xe[q].i1);
          b0[q] = __ldg(r01 + xe[q].i0); b1[q] = __ldg(r01 + xe[q].i1);
          c0[q] = __ldg(r10 + xe[q].i0); c1[q] = __ldg(r10 + xe[q].i1);
          e0[q] = __ldg(r11 + xe[q].i0); e1[q] = __ldg(r11 + xe[q].i1);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int gx = gx0 + 32 * q + lane;
        const uint32_t any = __float_as_uint(a0[q]) | __float_as_uint(a1[q]) | __float_as_uint(b0[q]) |
                             __float_as_uint(b1[q]) | __float_as_uint(c0[q]) | __float_as_uint(c1[q]) |
                             __float_as_uint(e0[q]) | __float_as_uint(e1[q]);
        uint8_t u = 0;
        if (__ballot_sync(0xffffffffu, any != 0u) != 0u) {
          float v = id.w0 * (ih.w0 * (xe[q].w0 * a0[q] + xe[q].w1 * a1[q]) + ih.w1 * (xe[q].w0 * b0[q] + xe[q].w1 * b1[q])) +
                    id.w1 * (ih.w0 * (xe[q].w0 * c0[q] + xe[q].w1 * c1[q]) + ih.w1 * (xe[q].w0 * e0[q] + xe[q].w1 * e1[q]));
          v = fminf(fmaxf(v, 0.0f), 1.0f);
          u = in[q] ? (uint8_t)(int)((double)v * 255.0) : 0;  // numpy: float64 product, astype(uint8) truncates
        }
        if (gx < OW) orow[gx] = u;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// Densitometry on the full-resolution grid: voxels per label, and per-slot HU histograms + exact HU sums.
// A thread takes DENS_VECS 16-voxel vectors per trip (grid-stride).  Runs of equal keys in the order a thread
// visits its voxels (label; or slot and bin) are folded into one shared atomic, and a run is carried across
// trips, so a thread that sees only background does one atomic in all.  Each CTA adds its nonzero shared
// counters into the int64 outputs with integer atomics: exact, whatever the order.
// ---------------------------------------------------------------------------------------
static constexpr int DENS_THREADS = 512;
static constexpr int DENS_VECS = 4;
static constexpr int HIST_VECS = 2;
static constexpr int DENS_LABELS = 256;
static constexpr int HU_BINS = 2048;
static constexpr int HU_LO = -1024;
static constexpr int HU_SLOTS = 16;
static constexpr unsigned NO_SLOT = 0xFFu;

struct SlotTable {
  uint8_t slot[DENS_LABELS];
};

// 16 labels of vector v as four little-endian words; zeros past the end of the volume.  nv: voxels in the vector.
template <bool VEC>
__device__ __forceinline__ int load_labels16(const uint8_t *__restrict__ lb, int64_t v, int64_t count, uint32_t (&w)[4]) {
  const int64_t o = v * 16, left = count - o;
  const int nv = left <= 0 ? 0 : (left >= 16 ? 16 : (int)left);
  if (VEC && nv == 16) {
    const uint4 q = __ldg(reinterpret_cast<const uint4 *>(lb + o));
    w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
  } else {
    w[0] = w[1] = w[2] = w[3] = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < nv) w[k >> 2] |= (uint32_t)__ldg(lb + o + k) << (8 * (k & 3));
  }
  return nv;
}

__device__ __forceinline__ unsigned byte16(const uint32_t (&w)[4], int k) { return (w[k >> 2] >> (8 * (k & 3))) & 0xffu; }

template <bool VEC>
__global__ void __launch_bounds__(DENS_THREADS)
label_counts_kernel(const uint8_t *__restrict__ labels, int64_t count, unsigned long long *__restrict__ counts) {
  __shared__ uint32_t cnt[DENS_LABELS];
  for (int i = threadIdx.x; i < DENS_LABELS; i += DENS_THREADS) cnt[i] = 0;
  __syncthreads();
  const int64_t vecs = (count + 15) / 16;
  const int64_t stride = (int64_t)gridDim.x * DENS_THREADS * DENS_VECS;
  unsigned cur = 0, run = 0;
  for (int64_t v0 = (int64_t)blockIdx.x * DENS_THREADS * DENS_VECS + threadIdx.x; v0 < vecs; v0 += stride) {
    uint32_t w[DENS_VECS][4];
    int nv[DENS_VECS];
#pragma unroll
    for (int j = 0; j < DENS_VECS; ++j) nv[j] = load_labels16<VEC>(labels, v0 + j * DENS_THREADS, count, w[j]);
#pragma unroll
    for (int j = 0; j < DENS_VECS; ++j) {
      const uint32_t rep = (w[j][0] & 0xffu) * 0x01010101u;
      if (nv[j] == 16 && w[j][0] == rep && w[j][1] == rep && w[j][2] == rep && w[j][3] == rep) {  // one label
        const unsigned lab = rep & 0xffu;
        if (lab != cur) {
          if (run) atomicAdd(&cnt[cur], run);
          cur = lab;
          run = 0;
        }
        run += 16;
        continue;
      }
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        if (k >= nv[j]) break;
        const unsigned lab = byte16(w[j], k);
        if (lab != cur) {
          if (run) atomicAdd(&cnt[cur], run);
          cur = lab;
          run = 0;
        }
        ++run;
      }
    }
  }
  if (run) atomicAdd(&cnt[cur], run);
  __syncthreads();
  for (int i = threadIdx.x; i < DENS_LABELS; i += DENS_THREADS)
    if (cnt[i]) atomicAdd(&counts[i], (unsigned long long)cnt[i]);
}

// Dynamic shared memory: nslots x 2048 uint32 bins (up to 128 KB).  The vector path keeps to 64 registers, so that two
// CTAs fit an SM whenever their bins do (the byte path, for unaligned views only, would spill there).
template <bool VEC>
__global__ void __launch_bounds__(DENS_THREADS, VEC ? 2 : 1)
label_hu_hist_kernel(const int16_t *__restrict__ scan, const uint8_t *__restrict__ labels, int64_t count,
                     const SlotTable table, int nslots, unsigned long long *__restrict__ hist,
                     unsigned long long *__restrict__ hu_sum) {
  extern __shared__ uint4 bins_raw[];
  uint32_t *bins = reinterpret_cast<uint32_t *>(bins_raw);
  __shared__ uint8_t slot_of[DENS_LABELS];
  __shared__ unsigned long long ssum[HU_SLOTS];
  const int nbins = nslots * HU_BINS;
  for (int i = threadIdx.x; i < nbins / 4; i += DENS_THREADS) bins_raw[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < DENS_LABELS; i += DENS_THREADS) slot_of[i] = table.slot[i];
  if (threadIdx.x < HU_SLOTS) ssum[threadIdx.x] = 0ull;
  __syncthreads();
  const bool zero_tracked = table.slot[0] != NO_SLOT;  // label 0 fills most of a chest scan: usually untracked
  const int64_t vecs = (count + 15) / 16;
  const int64_t stride = (int64_t)gridDim.x * DENS_THREADS * HIST_VECS;
  unsigned key = 0, krun = 0;        // run of one (slot, bin): bins[key] += krun
  unsigned scur = NO_SLOT;           // run of one slot: ssum[scur] += srun
  long long srun = 0;
  for (int64_t v0 = (int64_t)blockIdx.x * DENS_THREADS * HIST_VECS + threadIdx.x; v0 < vecs; v0 += stride) {
    uint32_t sw[HIST_VECS][4];       // labels, then their slots (NO_SLOT past the end)
    int nv[HIST_VECS];
    bool tracked[HIST_VECS];
#pragma unroll
    for (int j = 0; j < HIST_VECS; ++j) nv[j] = load_labels16<VEC>(labels, v0 + j * DENS_THREADS, count, sw[j]);
#pragma unroll
    for (int j = 0; j < HIST_VECS; ++j) {
      tracked[j] = false;
      if (nv[j] == 0 || (!zero_tracked && (sw[j][0] | sw[j][1] | sw[j][2] | sw[j][3]) == 0u)) continue;
      uint32_t s4[4] = {0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const unsigned s = k < nv[j] ? (unsigned)slot_of[byte16(sw[j], k)] : NO_SLOT;
        tracked[j] |= s != NO_SLOT;
        s4[k >> 2] |= s << (8 * (k & 3));
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) sw[j][q] = s4[q];
    }
    // the HU of every whole tracked vector of the trip, loaded before any is used (the byte path loads per voxel)
    uint4 hu[HIST_VECS][2];
#pragma unroll
    for (int j = 0; j < HIST_VECS; ++j) {
      hu[j][0] = hu[j][1] = make_uint4(0, 0, 0, 0);
      if (VEC && tracked[j] && nv[j] == 16) {
        const uint4 *p = reinterpret_cast<const uint4 *>(scan + (v0 + j * DENS_THREADS) * 16);
        hu[j][0] = __ldg(p);
        hu[j][1] = __ldg(p + 1);
      }
    }
#pragma unroll
    for (int j = 0; j < HIST_VECS; ++j) {
      if (!tracked[j]) continue;
      const bool whole = VEC && nv[j] == 16;
      const int16_t *sp = scan + (v0 + j * DENS_THREADS) * 16;
      const uint32_t hw[8] = {hu[j][0].x, hu[j][0].y, hu[j][0].z, hu[j][0].w,
                              hu[j][1].x, hu[j][1].y, hu[j][1].z, hu[j][1].w};
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const unsigned s = byte16(sw[j], k);
        if (s == NO_SLOT) continue;  // also every voxel past the end of the volume
        const int h = whole ? (int)(short)(uint16_t)(hw[k >> 1] >> (16 * (k & 1))) : (int)__ldg(sp + k);
        const unsigned b = (unsigned)(min(max(h, HU_LO), HU_LO + HU_BINS - 1) - HU_LO);
        const unsigned kk = s * HU_BINS + b;
        if (kk != key) {
          if (krun) atomicAdd(&bins[key], krun);
          key = kk;
          krun = 0;
        }
        ++krun;
        if (s != scur) {
          if (scur != NO_SLOT) atomicAdd(&ssum[scur], (unsigned long long)srun);
          scur = s;
          srun = 0;
        }
        srun += h;
      }
    }
  }
  if (krun) atomicAdd(&bins[key], krun);
  if (scur != NO_SLOT) atomicAdd(&ssum[scur], (unsigned long long)srun);
  __syncthreads();
  for (int i = threadIdx.x; i < nbins; i += DENS_THREADS)
    if (bins[i]) atomicAdd(&hist[i], (unsigned long long)bins[i]);
  if (threadIdx.x < nslots && ssum[threadIdx.x]) atomicAdd(&hu_sum[threadIdx.x], ssum[threadIdx.x]);
}

}  // namespace dram

using namespace dram;

static const int kThreads = 256;

extern "C" int dram_mask_bbox(const uint8_t *mask, int32_t D, int32_t H, int32_t W, int32_t *bbox, void *stream) {
  DRAM_REQUIRE(mask && bbox, "dram_mask_bbox: null pointer");
  DRAM_REQUIRE(D > 0 && H > 0 && W > 0 && (int64_t)D * H < 0x7fffffffLL, "dram_mask_bbox: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  bbox_init_kernel<<<1, 1, 0, st>>>(bbox, D, H, W);
  DRAM_CHECK_LAUNCH("bbox_init_kernel");
  mask_bbox_kernel<<<stream_grid((int64_t)D * H * 32, kThreads, 8), kThreads, 0, st>>>(mask, bbox, D, H, W);
  DRAM_CHECK_LAUNCH("mask_bbox_kernel");
  return DRAM_OK;
}

extern "C" size_t dram_lung_crop_workspace_bytes(int32_t cd, int32_t ch, int32_t cw) {
  if (cd <= 0 || ch <= 0 || cw <= 0) return 0;
  const BitWindow bw = bit_window(cd, ch, cw);  // two bit windows: lobe > 0, and its in-plane 5x5 maximum
  return 2 * (size_t)bw.wd * (size_t)bw.wh * (size_t)bw.ww * sizeof(uint32_t);
}

extern "C" int dram_lung_crop(const int16_t *scan, const uint8_t *lobe, int32_t D, int32_t H, int32_t W, int32_t z0,
                              int32_t y0, int32_t x0, int32_t cd, int32_t ch, int32_t cw, int16_t *image_c,
                              uint8_t *lung_c, uint8_t *ess_c, void *workspace, void *stream) {
  DRAM_REQUIRE(scan && lobe && image_c && lung_c && ess_c && workspace, "dram_lung_crop: null pointer");
  DRAM_REQUIRE(D > 0 && H > 0 && W > 0, "dram_lung_crop: empty volume");
  DRAM_REQUIRE(z0 >= 0 && y0 >= 0 && x0 >= 0 && cd > 0 && ch > 0 && cw > 0 && z0 + cd <= D && y0 + ch <= H &&
                   x0 + cw <= W,
               "dram_lung_crop: crop [%d:%d, %d:%d, %d:%d] outside the %dx%dx%d volume", z0, z0 + cd, y0, y0 + ch, x0,
               x0 + cw, D, H, W);
  cudaStream_t st = (cudaStream_t)stream;
  const BitWindow bw = bit_window(cd, ch, cw);
  const int64_t words = (int64_t)bw.wd * bw.wh * bw.ww;
  DRAM_REQUIRE((int64_t)bw.wd * bw.wh < 0x7fffffffLL, "dram_lung_crop: crop too large");
  uint32_t *bits = reinterpret_cast<uint32_t *>(workspace), *dil = bits + words;
  lung_pack_bits_kernel<<<stream_grid((int64_t)bw.wd * bw.wh * 32, kThreads, 8), kThreads, 0, st>>>(lobe, bits, D, H, W, z0,
                                                                                                  y0, x0, cd, ch, cw);
  DRAM_CHECK_LAUNCH("lung_pack_bits_kernel");
  lung_dilate_bits_kernel<<<stream_grid(words, kThreads), kThreads, 0, st>>>(bits, dil, cd, ch, cw);
  DRAM_CHECK_LAUNCH("lung_dilate_bits_kernel");
  const int64_t groups = ((int64_t)cd * ch * cw + 7) / 8;
  const int vec_ok = (reinterpret_cast<uintptr_t>(image_c) % 16 == 0) && (reinterpret_cast<uintptr_t>(lung_c) % 8 == 0) &&
                     (reinterpret_cast<uintptr_t>(ess_c) % 8 == 0);
  lung_crop_kernel<<<stream_grid(groups, kThreads), kThreads, 0, st>>>(scan, lobe, dil, image_c, lung_c, ess_c, D, H, W, z0,
                                                                      y0, x0, cd, ch, cw, (short)-2048, (short)-910, vec_ok);
  DRAM_CHECK_LAUNCH("lung_crop_kernel");
  return DRAM_OK;
}

extern "C" int dram_heatmap_u8(const float *map, int32_t d, int32_t h, int32_t w, uint8_t *out, int32_t OD, int32_t OH,
                               int32_t OW, int32_t z0, int32_t y0, int32_t x0, int32_t cd, int32_t ch, int32_t cw,
                               void *stream) {
  DRAM_REQUIRE(map && out, "dram_heatmap_u8: null pointer");
  DRAM_REQUIRE(d > 0 && h > 0 && w > 0 && OD > 0 && OH > 0 && OW > 0 && (int64_t)OD * OH < 0x7fffffffLL,
               "dram_heatmap_u8: bad shape");
  DRAM_REQUIRE(z0 >= 0 && y0 >= 0 && x0 >= 0 && cd > 0 && ch > 0 && cw > 0 && z0 + cd <= OD && y0 + ch <= OH &&
                   x0 + cw <= OW,
               "dram_heatmap_u8: crop outside the output volume");
  DRAM_REQUIRE((size_t)cw * sizeof(XEntry) <= 48 * 1024, "dram_heatmap_u8: crop wider than 3072 voxels");
  heatmap_u8_kernel<<<stream_grid((int64_t)OD * OH * 32, kThreads, 8), kThreads, (size_t)cw * sizeof(XEntry),
                      (cudaStream_t)stream>>>(
      map, out, d, h, w, OD, OH, OW, z0, y0, x0, cd, ch, cw, ac_scale(d, cd), ac_scale(h, ch), ac_scale(w, cw));
  DRAM_CHECK_LAUNCH("heatmap_u8_kernel");
  return DRAM_OK;
}

// Grid of the densitometry passes: enough CTAs to fill the device, no more than there are trips.
static int dens_grid(int64_t count, int vecs_per_trip, int ctas_per_sm) {
  const int64_t trips = ceil_div64(ceil_div64(count, 16), (int64_t)DENS_THREADS * vecs_per_trip);
  const int64_t cap = (int64_t)sm_count() * (ctas_per_sm < 1 ? 1 : ctas_per_sm);
  return (int)(trips < 1 ? 1 : (trips < cap ? trips : cap));
}

extern "C" int dram_label_counts(const uint8_t *labels, int64_t count, int64_t *counts, void *stream) {
  DRAM_REQUIRE(labels && counts, "dram_label_counts: null pointer");
  DRAM_REQUIRE(count >= 0 && count < 0x7fffffffLL, "dram_label_counts: count %lld outside 0 .. 2^31-1",
               (long long)count);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_cuda(cudaMemsetAsync(counts, 0, DENS_LABELS * sizeof(int64_t), st), "dram_label_counts: zeroing");
  if (rc != DRAM_OK || count == 0) return rc;
  unsigned long long *out = reinterpret_cast<unsigned long long *>(counts);
  if ((uintptr_t)labels % 16 == 0)
    label_counts_kernel<true><<<dens_grid(count, DENS_VECS, 4), DENS_THREADS, 0, st>>>(labels, count, out);
  else
    label_counts_kernel<false><<<dens_grid(count, DENS_VECS, 4), DENS_THREADS, 0, st>>>(labels, count, out);
  DRAM_CHECK_LAUNCH("label_counts_kernel");
  return DRAM_OK;
}

// CTAs of the histogram kernel per SM for `nslots` slots.  The shared-memory attribute and the occupancy query run on the
// first call per device and slot count only, so that later calls (e.g. under stream capture) make no such API call.
template <bool VEC>
static int hu_hist_ctas_per_sm(int nslots, int *per_sm) {
  static std::atomic<int> known[64][HU_SLOTS + 1];
  int dev = 0;
  int rc = check_cuda(cudaGetDevice(&dev), "dram_label_hu_hist: device");
  if (rc != DRAM_OK) return rc;
  if (dev >= 0 && dev < 64 && (*per_sm = known[dev][nslots].load()) > 0) return DRAM_OK;
  auto kernel = label_hu_hist_kernel<VEC>;
  rc = check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       HU_SLOTS * HU_BINS * (int)sizeof(uint32_t)),
                  "dram_label_hu_hist: shared memory attribute");
  if (rc != DRAM_OK) return rc;
  rc = check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kernel, DENS_THREADS,
                                                                 (size_t)nslots * HU_BINS * sizeof(uint32_t)),
                  "dram_label_hu_hist: occupancy");
  if (rc != DRAM_OK) return rc;
  if (*per_sm < 1) *per_sm = 1;
  if (dev >= 0 && dev < 64) known[dev][nslots].store(*per_sm);
  return DRAM_OK;
}

template <bool VEC>
static int launch_hu_hist(const int16_t *scan, const uint8_t *labels, int64_t count, const SlotTable &table,
                          int nslots, unsigned long long *hist, unsigned long long *hu_sum, cudaStream_t st) {
  int per_sm = 0;
  int rc = hu_hist_ctas_per_sm<VEC>(nslots, &per_sm);
  if (rc != DRAM_OK) return rc;
  label_hu_hist_kernel<VEC><<<dens_grid(count, HIST_VECS, per_sm), DENS_THREADS,
                              (size_t)nslots * HU_BINS * sizeof(uint32_t), st>>>(scan, labels, count, table, nslots,
                                                                                 hist, hu_sum);
  DRAM_CHECK_LAUNCH("label_hu_hist_kernel");
  return DRAM_OK;
}

extern "C" int dram_label_hu_hist(const int16_t *scan, const uint8_t *labels, int64_t count,
                                  const uint8_t *slot_of_label, int32_t nslots, int64_t *hist, int64_t *hu_sum,
                                  void *stream) {
  DRAM_REQUIRE(scan && labels && slot_of_label && hist && hu_sum, "dram_label_hu_hist: null pointer");
  DRAM_REQUIRE(nslots >= 1 && nslots <= HU_SLOTS, "dram_label_hu_hist: nslots %d outside 1..%d", nslots, HU_SLOTS);
  DRAM_REQUIRE(count >= 0 && count < 0x7fffffffLL, "dram_label_hu_hist: count %lld outside 0 .. 2^31-1",
               (long long)count);
  SlotTable table;
  for (int k = 0; k < DENS_LABELS; ++k) {
    DRAM_REQUIRE(slot_of_label[k] < nslots || slot_of_label[k] == NO_SLOT,
                 "dram_label_hu_hist: label %d goes to slot %d of %d", k, (int)slot_of_label[k], nslots);
    table.slot[k] = slot_of_label[k];
  }
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_cuda(cudaMemsetAsync(hist, 0, (size_t)nslots * HU_BINS * sizeof(int64_t), st),
                      "dram_label_hu_hist: zeroing");
  if (rc == DRAM_OK) rc = check_cuda(cudaMemsetAsync(hu_sum, 0, (size_t)nslots * sizeof(int64_t), st),
                                     "dram_label_hu_hist: zeroing");
  if (rc != DRAM_OK || count == 0) return rc;
  unsigned long long *h = reinterpret_cast<unsigned long long *>(hist), *s = reinterpret_cast<unsigned long long *>(hu_sum);
  if (((uintptr_t)scan | (uintptr_t)labels) % 16 == 0) return launch_hu_hist<true>(scan, labels, count, table, nslots, h, s, st);
  return launch_hu_hist<false>(scan, labels, count, table, nslots, h, s, st);
}
