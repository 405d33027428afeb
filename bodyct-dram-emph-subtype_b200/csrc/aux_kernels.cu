// Memory-bound kernels of the hot path (K2a, K3, K4, K6, K7, K8, K8b + layout helpers).
// All are grid-stride kernels with 16-byte vector accesses on the contiguous (channel or W)
// axis and grids sized as a multiple of the SM count; none has data reuse worth staging in
// shared memory beyond what L1/L2 already give (each input element is touched by <= 27
// neighbouring outputs that sit in the same or the adjacent CTA).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "common.h"

namespace dram {

typedef __nv_bfloat16 bf16;
typedef __nv_bfloat162 bf162;

// Two packed 16-bit activations <-> fp32 for either storage type (f16 != 0: IEEE half, else bf16).
__device__ __forceinline__ uint32_t pack2(float a, float b, int f16) {
  if (f16) {  // saturating conversion (F2FP.SATFINITE), no inf
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
  bf162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t *>(&h);
}
__device__ __forceinline__ float2 unpack2(uint32_t u, int f16) {
  if (f16) return __half22float2(*reinterpret_cast<__half2 *>(&u));
  bf162 h = *reinterpret_cast<bf162 *>(&u);
  return make_float2(__low2float(h), __high2float(h));
}
__device__ __forceinline__ float load16(const uint16_t *p, int f16) {
  return f16 ? __half2float(*reinterpret_cast<const __half *>(p)) : __bfloat162float(*reinterpret_cast<const bf16 *>(p));
}
__device__ __forceinline__ uint16_t store16(float v, int f16) {
  if (f16) {
    __half h = __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
    return *reinterpret_cast<uint16_t *>(&h);
  }
  bf16 h = __float2bfloat16_rn(v);
  return *reinterpret_cast<uint16_t *>(&h);
}

// ATen's legacy `nearest` source index (nearest_idx in UpSample.h).
__device__ __forceinline__ int nearest_index(int dst, int in_size, int out_size) {
  if (out_size == in_size) return dst;
  if (out_size == 2 * in_size) return dst >> 1;
  const float scale = (float)in_size / (float)out_size;
  const int s = (int)floorf((float)dst * scale);
  return s < in_size - 1 ? s : in_size - 1;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Block-wide sums of `a` and `b` in one pair of barriers; results valid in thread 0.
__device__ __forceinline__ void block_sum2(double &a, double &b, double2 *scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  a = warp_sum(a);
  b = warp_sum(b);
  __syncthreads();
  if (lane == 0) scratch[warp] = make_double2(a, b);
  __syncthreads();
  if (warp == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    const double2 v = lane < nw ? scratch[lane] : make_double2(0.0, 0.0);
    a = warp_sum(v.x);
    b = warp_sum(v.y);
  }
}
// Block-wide sum of `v`; result valid in thread 0.  `scratch` has >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double *scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  if (warp == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    v = lane < nw ? scratch[lane] : 0.0;
    v = warp_sum(v);
  }
  return v;
}

// ---------------------------------------------------------------------------------------
// K2a stem unfold: one 16-byte store per thread (8 pseudo-channels = one kh row of taps).
// ---------------------------------------------------------------------------------------
__global__ void stem_expand_kernel(const float *__restrict__ x, uint4 *__restrict__ out, int n, int d,
                                   int h, int w, int h2, int w2, int f16) {
  const int64_t total = (int64_t)n * d * h2 * w2 * 8;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int kh = (int)(t & 7);
    int64_t v = t >> 3;
    const int ow = (int)(v % w2);
    v /= w2;
    const int oh = (int)(v % h2);
    v /= h2;  // v = n*d + z
    const int ih = 2 * oh - 3 + kh;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = 0.0f;
    if (kh < 7 && ih >= 0 && ih < h) {
      const float *row = x + (v * h + ih) * (int64_t)w;
      const int iw0 = 2 * ow - 3;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const int iw = iw0 + j;
        if (iw >= 0 && iw < w) f[j] = __ldg(row + iw);
      }
    }
    out[t] = make_uint4(pack2(f[0], f[1], f16), pack2(f[2], f[3], f16), pack2(f[4], f[5], f16),
                        pack2(f[6], f[7], f16));
  }
}

// ---------------------------------------------------------------------------------------
// K3 max-pool 3^3 s2 p1, NDHWC 16-bit, 8 channels per thread.  A thread owns one (h, w, channel
// group) of the output and marches over a chunk of output planes: the 3x3 in-plane maximum of input
// plane 2d+1 is the first plane of the next window too, so each output costs 18 instead of 27
// 16-byte loads.  Out-of-range taps are clamped instead of skipped (the clamped voxel always lies
// inside the window, so the maximum is unchanged): every load is unconditional and the 9 loads of
// a plane are in flight together.
// ---------------------------------------------------------------------------------------
static constexpr int POOL_DCHUNK = 8;

template <bool F16>
__device__ __forceinline__ void max8(uint4 &m, const uint4 u) {
  if constexpr (F16) {
    __half2 *a = reinterpret_cast<__half2 *>(&m);
    const __half2 *b = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
    for (int q = 0; q < 4; ++q) a[q] = __hmax2(a[q], b[q]);
  } else {
    bf162 *a = reinterpret_cast<bf162 *>(&m);
    const bf162 *b = reinterpret_cast<const bf162 *>(&u);
#pragma unroll
    for (int q = 0; q < 4; ++q) a[q] = __hmax2(a[q], b[q]);
  }
}

template <bool F16>
__global__ void __launch_bounds__(256, 3)
maxpool3d_kernel(const uint4 *__restrict__ x, uint4 *__restrict__ out, int n, int d, int h, int w, int cg,
                 int od, int oh, int ow, int dchunks) {
  const int64_t total = (int64_t)n * dchunks * oh * ow * cg;
  const int row = w * cg;
  const int64_t plane = (int64_t)h * row;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(t % cg);
    int64_t v = t / cg;
    const int xw = (int)(v % ow);
    v /= ow;
    const int xh = (int)(v % oh);
    v /= oh;
    const int ck = (int)(v % dchunks);
    const int b = (int)(v / dchunks);
    int off[9];  // in-plane offsets of the 3x3 window (clamped taps repeat a voxel of the window)
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int c = 0; c < 3; ++c)
        off[a * 3 + c] = min(max(2 * xh - 1 + a, 0), h - 1) * row + min(max(2 * xw - 1 + c, 0), w - 1) * cg + g;
    const uint4 *xb = x + (int64_t)b * d * plane;
    auto plane_max = [&](int z) {
      const uint4 *p = xb + (int64_t)min(max(z, 0), d - 1) * plane;
      uint4 u[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) u[i] = __ldg(p + off[i]);
      uint4 m = u[0];
#pragma unroll
      for (int i = 1; i < 9; ++i) max8<F16>(m, u[i]);
      return m;
    };
    const int xd0 = ck * POOL_DCHUNK, xd1 = min(od, xd0 + POOL_DCHUNK);
    uint4 carry = plane_max(2 * xd0 - 1);
    uint4 *o = out + ((((int64_t)b * od + xd0) * oh + xh) * ow + xw) * cg + g;
    const int64_t ostride = (int64_t)oh * ow * cg;
    for (int xd = xd0; xd < xd1; ++xd) {
      uint4 m = carry;
      max8<F16>(m, plane_max(2 * xd));
      carry = plane_max(2 * xd + 1);
      max8<F16>(m, carry);
      *o = m;
      o += ostride;
    }
  }
}

// ---------------------------------------------------------------------------------------
// K4 trilinear x2 (align_corners=True), NDHWC 16-bit, 8 channels per thread, fp32 math in ATen's
// nesting order (W innermost, D outermost).  A thread owns one (h, w, channel group) of the output
// and marches over a chunk of output planes; the in-plane bilinear combinations of the two
// bracketing input planes stay in registers, and because the source step (d-1)/(2d-1) is below one
// half the lower plane advances by at most one per output: ~2.5 instead of 8 16-byte loads per
// output, and the storage type is a template parameter (no per-value type branches).
// ---------------------------------------------------------------------------------------
static constexpr int UP_DCHUNK = 8;

template <bool F16>
__device__ __forceinline__ float2 unpack2t(uint32_t u) {
  if constexpr (F16) return __half22float2(*reinterpret_cast<const __half2 *>(&u));
  // bf16 -> fp32 is a 16-bit shift
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}
template <bool F16>
__device__ __forceinline__ uint32_t pack2t(float a, float b) {
  if constexpr (F16) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  } else {
    const bf162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&h);
  }
}

template <bool F16>
__global__ void __launch_bounds__(256, 3)
upsample2x_kernel(const uint4 *__restrict__ x, uint4 *__restrict__ out, int n, int d, int h, int w, int cg,
                  float sd, float sh, float sw, int dchunks) {
  const int od = 2 * d, oh = 2 * h, ow = 2 * w;
  const int64_t total = (int64_t)n * dchunks * oh * ow * cg;
  const int64_t plane = (int64_t)h * w * cg;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(t % cg);
    int64_t v = t / cg;
    const int xw = (int)(v % ow);
    v /= ow;
    const int xh = (int)(v % oh);
    v /= oh;
    const int ck = (int)(v % dchunks);
    const int b = (int)(v / dchunks);
    const LinIdx ih = lin_index_ac(xh, sh, h), iw = lin_index_ac(xw, sw, w);
    const int o00 = (ih.i0 * w + iw.i0) * cg + g, o01 = (ih.i0 * w + iw.i1) * cg + g;
    const int o10 = (ih.i1 * w + iw.i0) * cg + g, o11 = (ih.i1 * w + iw.i1) * cg + g;
    const uint4 *xb = x + (int64_t)b * d * plane;
    // in-plane bilinear combination of input plane z: h0*(w0*a + w1*b) + h1*(w0*c + w1*d)
    auto plane_val = [&](int z, float (&P)[8]) {
      const uint4 *p = xb + (int64_t)z * plane;
      const uint4 ua = __ldg(p + o00), ub = __ldg(p + o01), uc = __ldg(p + o10), ud = __ldg(p + o11);
      const uint32_t a_[4] = {ua.x, ua.y, ua.z, ua.w}, b_[4] = {ub.x, ub.y, ub.z, ub.w};
      const uint32_t c_[4] = {uc.x, uc.y, uc.z, uc.w}, d_[4] = {ud.x, ud.y, ud.z, ud.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 fa = unpack2t<F16>(a_[q]), fb = unpack2t<F16>(b_[q]), fc = unpack2t<F16>(c_[q]),
                     fd = unpack2t<F16>(d_[q]);
        P[2 * q + 0] = bilerp_hw(fa.x, fb.x, fc.x, fd.x, iw.w0, iw.w1, ih.w0, ih.w1);
        P[2 * q + 1] = bilerp_hw(fa.y, fb.y, fc.y, fd.y, iw.w0, iw.w1, ih.w0, ih.w1);
      }
    };
    const int xd0 = ck * UP_DCHUNK, xd1 = min(od, xd0 + UP_DCHUNK);
    float P0[8], P1[8];
    int cur = lin_index_ac(xd0, sd, d).i0;
    plane_val(cur, P0);
    plane_val(min(cur + 1, d - 1), P1);
    uint4 *o = out + ((((int64_t)b * od + xd0) * oh + xh) * ow + xw) * cg + g;
    const int64_t ostride = (int64_t)oh * ow * cg;
    for (int xd = xd0; xd < xd1; ++xd) {
      const LinIdx id = lin_index_ac(xd, sd, d);
      if (id.i0 != cur) {  // the lower plane moved up by one: the old upper plane becomes the lower one
        cur = id.i0;
#pragma unroll
        for (int j = 0; j < 8; ++j) P0[j] = P1[j];
        if (cur + 1 < d) plane_val(cur + 1, P1);  // at the last plane i1 == i0 and P1 == P0 already
      }
      float o8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o8[j] = lerp_d(P0[j], P1[j], id.w0, id.w1);
      *o = make_uint4(pack2t<F16>(o8[0], o8[1]), pack2t<F16>(o8[2], o8[3]), pack2t<F16>(o8[4], o8[5]),
                      pack2t<F16>(o8[6], o8[7]));
      o += ostride;
    }
  }
}

// ---------------------------------------------------------------------------------------
// K6 lobe-masked (or plain) mean of each dense channel.
// grid = (blocks, ch, n); one warp per (d, h) row of the map, so the row's mask indices are decoded
// once and the lanes stream the row with 16-byte loads (VEC = 4) when w % 4 == 0.
// sums: double [n][ch+1] (last slot = sum of mask / voxel count).
// ---------------------------------------------------------------------------------------
template <typename MaskT, int VEC>
__global__ void __launch_bounds__(256)
masked_pool_partial_kernel(const float *__restrict__ dense, const MaskT *__restrict__ mask,
                           double *__restrict__ sums, int ch, int d, int h, int w, int md, int mh, int mw) {
  __shared__ double scratch[32];
  const int c = blockIdx.y, b = blockIdx.z;
  const int64_t plane = (int64_t)d * h * w;
  const float *src = dense + ((int64_t)b * ch + c) * plane;
  const MaskT *mk = mask ? mask + (int64_t)b * md * mh * mw : nullptr;
  const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  const int rows = d * h, wv = w / VEC;
  double s = 0.0, ms = 0.0;
  for (int r = blockIdx.x * warps + (threadIdx.x >> 5); r < rows; r += gridDim.x * warps) {
    const int xd = r / h, xh = r - xd * h;
    const float *row = src + (int64_t)r * w;
    const MaskT *mrow = nullptr;
    if (mk) mrow = mk + ((int64_t)nearest_index(xd, md, d) * mh + nearest_index(xh, mh, h)) * mw;
    float fs = 0.0f, fm = 0.0f;  // a row chunk per lane: at most a few hundred values in [0,1]-ish range
    for (int xv = lane; xv < wv; xv += 32) {
      float v[VEC];
      if constexpr (VEC == 4) {
        const float4 f = __ldg(reinterpret_cast<const float4 *>(row) + xv);
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
      } else {
        v[0] = __ldg(row + xv);
      }
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        float m = 1.0f;
        if (mrow) {
          const MaskT mv = mrow[nearest_index(xv * VEC + j, mw, w)];
          if constexpr (sizeof(MaskT) == 1) m = mv ? 1.0f : 0.0f;
          else m = (float)mv;  // float lungs are used as weights, exactly like `dout * lungs` (med3d.py:387)
        }
        fs += v[j] * m;
        fm += m;
      }
    }
    s += (double)fs;
    ms += (double)fm;
  }
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[(int64_t)b * (ch + 1) + c], s);
  if (c == 0) {
    ms = block_sum(ms, scratch);
    if (threadIdx.x == 0) atomicAdd(&sums[(int64_t)b * (ch + 1) + ch], ms);
  }
}
__global__ void masked_pool_finalize_kernel(const double *__restrict__ sums, float *__restrict__ out,
                                            int n, int ch) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * ch) return;
  const int b = i / ch, c = i % ch;
  out[i] = (float)sums[(int64_t)b * (ch + 1) + c] / (float)sums[(int64_t)b * (ch + 1) + ch];
}

// ---------------------------------------------------------------------------------------
// K7 dRAM: both maps in one pass.  One warp per output row (d, h): the D/H source planes and weights
// are decoded once per row; a lane produces 4 consecutive voxels along W per step when W % 4 == 0
// (float4 stores, uchar4 mask loads), one otherwise.  Voxels outside `ess` are exact zeros and cost
// no loads.  sums: double [2*n + n]: sum(out0[b]), sum(out1[b]), sum(lungs[b]).
// ---------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256)
dram_upsample_mask_kernel(const float *__restrict__ dense0, const float *__restrict__ dense1,
                          const uint8_t *__restrict__ ess, const uint8_t *__restrict__ lungs,
                          float *__restrict__ out0, float *__restrict__ out1, double *__restrict__ sums, int n,
                          int d, int h, int w, int D, int H, int W, float sd, float sh, float sw,
                          int blocks_per_sample) {
  __shared__ double scratch[32];
  const int b = blockIdx.x / blocks_per_sample;
  const int blk = blockIdx.x - b * blocks_per_sample;
  const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  const int Wv = W / VEC, rows = D * H;
  const int64_t splane = (int64_t)d * h * w;
  const float *s0 = dense0 + (int64_t)b * splane;
  const float *s1 = dense1 + (int64_t)b * splane;
  double acc0 = 0.0, acc1 = 0.0;
  unsigned lung_count = 0;
  for (int r = blk * warps + (threadIdx.x >> 5); r < rows; r += blocks_per_sample * warps) {
    const int xd = r / H, xh = r - xd * H;
    const LinIdx id = lin_index_ac(xd, sd, d), ih = lin_index_ac(xh, sh, h);
    const int r00 = (id.i0 * h + ih.i0) * w, r01 = (id.i0 * h + ih.i1) * w;
    const int r10 = (id.i1 * h + ih.i0) * w, r11 = (id.i1 * h + ih.i1) * w;
    const int64_t obase = ((int64_t)b * rows + r) * W;
    for (int xv = lane; xv < Wv; xv += 32) {
      const int64_t o = obase + (int64_t)xv * VEC;
      uint8_t e[VEC], l[VEC];
      if constexpr (VEC == 4) {
        const uchar4 e4 = *reinterpret_cast<const uchar4 *>(ess + o);
        const uchar4 l4 = *reinterpret_cast<const uchar4 *>(lungs + o);
        e[0] = e4.x; e[1] = e4.y; e[2] = e4.z; e[3] = e4.w;
        l[0] = l4.x; l[1] = l4.y; l[2] = l4.z; l[3] = l4.w;
      } else {
        e[0] = ess[o];
        l[0] = lungs[o];
      }
      float v0[VEC], v1[VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        float a = 0.0f, c = 0.0f;
        if (e[j]) {  // the product with ess == 0 is an exact 0 either way; skip the 16 loads
          const LinIdx iw = lin_index_ac(xv * VEC + j, sw, w);
          a = id.w0 * (ih.w0 * (iw.w0 * __ldg(s0 + r00 + iw.i0) + iw.w1 * __ldg(s0 + r00 + iw.i1)) +
                       ih.w1 * (iw.w0 * __ldg(s0 + r01 + iw.i0) + iw.w1 * __ldg(s0 + r01 + iw.i1))) +
              id.w1 * (ih.w0 * (iw.w0 * __ldg(s0 + r10 + iw.i0) + iw.w1 * __ldg(s0 + r10 + iw.i1)) +
                       ih.w1 * (iw.w0 * __ldg(s0 + r11 + iw.i0) + iw.w1 * __ldg(s0 + r11 + iw.i1)));
          c = id.w0 * (ih.w0 * (iw.w0 * __ldg(s1 + r00 + iw.i0) + iw.w1 * __ldg(s1 + r00 + iw.i1)) +
                       ih.w1 * (iw.w0 * __ldg(s1 + r01 + iw.i0) + iw.w1 * __ldg(s1 + r01 + iw.i1))) +
              id.w1 * (ih.w0 * (iw.w0 * __ldg(s1 + r10 + iw.i0) + iw.w1 * __ldg(s1 + r10 + iw.i1)) +
                       ih.w1 * (iw.w0 * __ldg(s1 + r11 + iw.i0) + iw.w1 * __ldg(s1 + r11 + iw.i1)));
          acc0 += (double)a;
          acc1 += (double)c;
        }
        v0[j] = a;
        v1[j] = c;
        lung_count += l[j] ? 1u : 0u;
      }
      if constexpr (VEC == 4) {
        *reinterpret_cast<float4 *>(out0 + o) = make_float4(v0[0], v0[1], v0[2], v0[3]);
        *reinterpret_cast<float4 *>(out1 + o) = make_float4(v1[0], v1[1], v1[2], v1[3]);
      } else {
        out0[o] = v0[0];
        out1[o] = v1[0];
      }
    }
  }
  acc0 = block_sum(acc0, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[b], acc0);
  acc1 = block_sum(acc1, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[n + b], acc1);
  double accl = block_sum((double)lung_count, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[2 * n + b], accl);
}

// ---------------------------------------------------------------------------------------
// K7, staged variant (the default): a CTA owns RH consecutive output rows of one output plane (b, xd, xh0..).
//   1. every thread loads the 16-voxel mask segments it owns (uint4 of ess + uint4 of lungs: 32 B in flight per
//      thread) — the dRAM is zero outside `ess`, which is ~2 % of a chest volume, so the kernel is a masked fill:
//      what bounds it is bytes in flight, not arithmetic;
//   2. if any voxel of the CTA's rows lies in `ess`, the half-resolution source brick those rows interpolate from
//      (2 planes x (RH/2 + 2) rows x w floats x 2 maps, <= 96*w bytes) is staged in shared memory with coalesced
//      16-byte loads, and the 2 x 8 gathers per voxel read shared memory instead of L1/L2;
//   3. results leave through 16-byte streaming stores (st.global.cs: the maps are not re-read by this kernel).
// The interpolation expression and its rounding order are those of the row kernel above (ATen's nesting).
// sums: double [3n] as above.  grid = (blocks per sample, n).
// ---------------------------------------------------------------------------------------
static constexpr int K7_SEG = 16;
static constexpr int K7_THREADS = 256;

__device__ __forceinline__ unsigned nonzero_bytes(uint32_t w) { return __vsadu4(__vsetne4(w, 0u), 0u); }

template <bool FAST>
__global__ void __launch_bounds__(K7_THREADS)
dram_upsample_mask_staged_kernel(const float *__restrict__ dense0, const float *__restrict__ dense1,
                                 const uint8_t *__restrict__ ess, const uint8_t *__restrict__ lungs,
                                 float *__restrict__ out0, float *__restrict__ out1, double *__restrict__ sums,
                                 int n, int d, int h, int w, int D, int H, int W, float sd, float sh, float sw,
                                 int RH, int nr_max) {
  extern __shared__ float k7_smem[];  // [map 2][plane 2][nr_max][w]
  __shared__ double scratch[32];
  const int b = blockIdx.y;
  const int segs = (W + K7_SEG - 1) / K7_SEG;
  const int hblocks = (H + RH - 1) / RH;
  const int groups = D * hblocks;
  const int items = RH * segs;
  const int64_t splane = (int64_t)d * h * w;
  const float *s0 = dense0 + (int64_t)b * splane;
  const float *s1 = dense1 + (int64_t)b * splane;
  const int64_t vol = (int64_t)D * H * W;
  const uint8_t *eb = ess + (int64_t)b * vol;
  const uint8_t *lb = lungs + (int64_t)b * vol;
  float *o0 = out0 + (int64_t)b * vol;
  float *o1 = out1 + (int64_t)b * vol;
  const int plane_stride = nr_max * w;  // floats per staged plane
  double acc0 = 0.0, acc1 = 0.0;
  unsigned lung_count = 0;

  for (int g = blockIdx.x; g < groups; g += gridDim.x) {
    const int xd = g / hblocks, xh0 = (g - xd * hblocks) * RH;
    const int rows = min(RH, H - xh0);
    const LinIdx id = lin_index_ac(xd, sd, d);
    const int ih_lo = lin_index_ac(xh0, sh, h).i0;
    const int ih_hi = lin_index_ac(xh0 + rows - 1, sh, h).i1;
    const int nr = ih_hi - ih_lo + 1;  // <= nr_max by construction (host)
    // ---- 1. masks of this thread's segments (at most 2 per thread: items <= 2 * K7_THREADS, host-checked)
    uint4 e4[2], l4[2];
    int any = 0;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int it = threadIdx.x + k * K7_THREADS;
      e4[k] = make_uint4(0, 0, 0, 0);
      l4[k] = make_uint4(0, 0, 0, 0);
      if (it < items) {
        const int r = it / segs, sg = it - r * segs;
        if (r < rows) {
          const int64_t o = ((int64_t)xd * H + xh0 + r) * W + (int64_t)sg * K7_SEG;
          if constexpr (FAST) {
            e4[k] = __ldcs(reinterpret_cast<const uint4 *>(eb + o));
            l4[k] = __ldcs(reinterpret_cast<const uint4 *>(lb + o));
          } else {
            uint8_t *ep = reinterpret_cast<uint8_t *>(&e4[k]), *lp = reinterpret_cast<uint8_t *>(&l4[k]);
            const int cnt = min(K7_SEG, W - sg * K7_SEG);
            for (int j = 0; j < cnt; ++j) {
              ep[j] = eb[o + j];
              lp[j] = lb[o + j];
            }
          }
          lung_count += nonzero_bytes(l4[k].x) + nonzero_bytes(l4[k].y) + nonzero_bytes(l4[k].z) + nonzero_bytes(l4[k].w);
          any |= (e4[k].x | e4[k].y | e4[k].z | e4[k].w) != 0;
        }
      }
    }
    // ---- 2. stage the source brick if anybody needs it (also orders the reuse of the buffer between groups)
    const int need = __syncthreads_or(any);
    if (need) {
      const int row_f4 = w >> 2;  // FAST implies w % 4 == 0 (host)
      if (FAST) {
        const int total = 4 * nr * row_f4;  // (map, plane, row, float4)
        for (int t = threadIdx.x; t < total; t += K7_THREADS) {
          const int c = t % row_f4;
          int q = t / row_f4;
          const int r = q % nr;
          q /= nr;
          const int pl = q & 1, mp = q >> 1;
          const float *src = (mp ? s1 : s0) + ((int64_t)(pl ? id.i1 : id.i0) * h + ih_lo + r) * w;
          reinterpret_cast<float4 *>(k7_smem + (mp * 2 + pl) * plane_stride + r * w)[c] =
              __ldg(reinterpret_cast<const float4 *>(src) + c);
        }
      } else {
        const int total = 4 * nr * w;
        for (int t = threadIdx.x; t < total; t += K7_THREADS) {
          const int c = t % w;
          int q = t / w;
          const int r = q % nr;
          q /= nr;
          const int pl = q & 1, mp = q >> 1;
          const float *src = (mp ? s1 : s0) + ((int64_t)(pl ? id.i1 : id.i0) * h + ih_lo + r) * w;
          k7_smem[(mp * 2 + pl) * plane_stride + r * w + c] = __ldg(src + c);
        }
      }
      __syncthreads();
    }
    // ---- 3. produce the segments
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int it = threadIdx.x + k * K7_THREADS;
      if (it >= items) continue;
      const int r = it / segs, sg = it - r * segs;
      if (r >= rows) continue;
      const int xh = xh0 + r, xw0 = sg * K7_SEG;
      const int64_t o = ((int64_t)xd * H + xh) * W + xw0;
      float v0[K7_SEG], v1[K7_SEG];
#pragma unroll
      for (int j = 0; j < K7_SEG; ++j) v0[j] = v1[j] = 0.0f;
      if ((e4[k].x | e4[k].y | e4[k].z | e4[k].w) != 0) {
        const LinIdx ih = lin_index_ac(xh, sh, h);
        const float *p00 = k7_smem + (ih.i0 - ih_lo) * w, *p01 = k7_smem + (ih.i1 - ih_lo) * w;
        const float *p10 = p00 + plane_stride, *p11 = p01 + plane_stride;
        const float *q00 = p00 + 2 * plane_stride, *q01 = p01 + 2 * plane_stride;
        const float *q10 = p10 + 2 * plane_stride, *q11 = p11 + 2 * plane_stride;
        const uint32_t ew[4] = {e4[k].x, e4[k].y, e4[k].z, e4[k].w};
#pragma unroll
        for (int j = 0; j < K7_SEG; ++j) {
          if ((ew[j >> 2] >> (8 * (j & 3))) & 0xffu) {
            const LinIdx iw = lin_index_ac(xw0 + j, sw, w);
            const float a = id.w0 * (ih.w0 * (iw.w0 * p00[iw.i0] + iw.w1 * p00[iw.i1]) +
                                     ih.w1 * (iw.w0 * p01[iw.i0] + iw.w1 * p01[iw.i1])) +
                            id.w1 * (ih.w0 * (iw.w0 * p10[iw.i0] + iw.w1 * p10[iw.i1]) +
                                     ih.w1 * (iw.w0 * p11[iw.i0] + iw.w1 * p11[iw.i1]));
            const float c = id.w0 * (ih.w0 * (iw.w0 * q00[iw.i0] + iw.w1 * q00[iw.i1]) +
                                     ih.w1 * (iw.w0 * q01[iw.i0] + iw.w1 * q01[iw.i1])) +
                            id.w1 * (ih.w0 * (iw.w0 * q10[iw.i0] + iw.w1 * q10[iw.i1]) +
                                     ih.w1 * (iw.w0 * q11[iw.i0] + iw.w1 * q11[iw.i1]));
            v0[j] = a;
            v1[j] = c;
            acc0 += (double)a;
            acc1 += (double)c;
          }
        }
      }
      if constexpr (FAST) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          __stcs(reinterpret_cast<float4 *>(o0 + o) + q, make_float4(v0[4 * q], v0[4 * q + 1], v0[4 * q + 2], v0[4 * q + 3]));
          __stcs(reinterpret_cast<float4 *>(o1 + o) + q, make_float4(v1[4 * q], v1[4 * q + 1], v1[4 * q + 2], v1[4 * q + 3]));
        }
      } else {
        const int cnt = min(K7_SEG, W - xw0);
        for (int j = 0; j < cnt; ++j) {
          o0[o + j] = v0[j];
          o1[o + j] = v1[j];
        }
      }
    }
  }
  acc0 = block_sum(acc0, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[b], acc0);
  acc1 = block_sum(acc1, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[n + b], acc1);
  double accl = block_sum((double)lung_count, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[2 * n + b], accl);
}

// ---------------------------------------------------------------------------------------
// K7, lean variant of the staged kernel for the common shapes (W a power-of-two multiple of 16 between 64 and 1024,
// w = W/2... any w % 4 == 0, everything 16-byte aligned).  Round-2 ncu: both K7 kernels moved their 168 MB at 13 % of
// the DRAM peak with no unit saturated — they were bound by instruction issue (index decoding with 64-bit divisions,
// two work items per thread, 32-element value arrays).  Here one CTA = one output plane slice of RY rows (grid =
// (H/RY, D, n): no division anywhere), thread (sx, ry) owns ONE 16-voxel segment: 2 x 16-byte mask loads, a block
// vote, and — for the ~90 % of CTAs without an `ess` voxel — eight 16-byte streaming stores of zeros and one integer
// warp reduction for the lung count.  CTAs that do meet `ess` stage the source brick in shared memory as before.
// ---------------------------------------------------------------------------------------
template <int LOG_SX>
__global__ void __launch_bounds__(256)
dram_upsample_mask_lean_kernel(const float *__restrict__ dense0, const float *__restrict__ dense1,
                               const uint8_t *__restrict__ ess, const uint8_t *__restrict__ lungs,
                               float *__restrict__ out0, float *__restrict__ out1, double *__restrict__ sums, int n,
                               int d, int h, int w, int D, int H, int W, float sd, float sh, float sw, int nr_max) {
  extern __shared__ __align__(128) float k7_smem[];  // [2 maps][4096] output staging, then [map 2][plane 2][nr_max][w]
  __shared__ double scratch[32];
  __shared__ unsigned lung_part[8];
  constexpr int SX = 1 << LOG_SX, RY = 256 >> LOG_SX;
  constexpr int SLICE = 256 * K7_SEG;                // RY rows x W voxels = 4096 floats = 16 KiB per map
  float *stage = k7_smem;
  float *brick = k7_smem + 2 * SLICE;
  const int sx = threadIdx.x & (SX - 1), ry = threadIdx.x >> LOG_SX;
  const int b = blockIdx.z, xd = blockIdx.y, xh0 = blockIdx.x * RY;
  const int xh = xh0 + ry;
  const bool row_ok = xh < H;
  const int64_t vol = (int64_t)D * H * W;
  const int64_t o = (int64_t)b * vol + ((int64_t)xd * H + xh) * W + sx * K7_SEG;
  uint4 e4 = make_uint4(0, 0, 0, 0), l4 = make_uint4(0, 0, 0, 0);
  if (row_ok) {
    e4 = __ldcs(reinterpret_cast<const uint4 *>(ess + o));
    l4 = __ldcs(reinterpret_cast<const uint4 *>(lungs + o));
  }
  const unsigned lung_count = nonzero_bytes(l4.x) + nonzero_bytes(l4.y) + nonzero_bytes(l4.z) + nonzero_bytes(l4.w);
  const int mine = (e4.x | e4.y | e4.z | e4.w) != 0;
  const int need = __syncthreads_or(mine);
  double acc0 = 0.0, acc1 = 0.0;
  float v0[K7_SEG], v1[K7_SEG];
#pragma unroll
  for (int j = 0; j < K7_SEG; ++j) v0[j] = v1[j] = 0.0f;
  if (need) {
    const LinIdx id = lin_index_ac(xd, sd, d);
    const int rows = min(RY, H - xh0);
    const int ih_lo = lin_index_ac(xh0, sh, h).i0;
    const int nr = lin_index_ac(xh0 + rows - 1, sh, h).i1 - ih_lo + 1;  // <= nr_max (host)
    const int plane_stride = nr_max * w;
    const float *s0 = dense0 + (int64_t)b * d * h * w, *s1 = dense1 + (int64_t)b * d * h * w;
    const int row_f4 = w >> 2, total = 4 * nr * row_f4;
    for (int t = threadIdx.x; t < total; t += 256) {
      const int c = t % row_f4;
      int q = t / row_f4;
      const int r = q % nr;
      q /= nr;
      const int pl = q & 1, mp = q >> 1;
      const float *src = (mp ? s1 : s0) + ((int64_t)(pl ? id.i1 : id.i0) * h + ih_lo + r) * w;
      reinterpret_cast<float4 *>(brick + (mp * 2 + pl) * plane_stride + r * w)[c] = __ldg(reinterpret_cast<const float4 *>(src) + c);
    }
    __syncthreads();
    if (mine) {
      const LinIdx ih = lin_index_ac(xh, sh, h);
      const float *p00 = brick + (ih.i0 - ih_lo) * w, *p01 = brick + (ih.i1 - ih_lo) * w;
      const float *p10 = p00 + plane_stride, *p11 = p01 + plane_stride;
      const float *q00 = p00 + 2 * plane_stride, *q01 = p01 + 2 * plane_stride;
      const float *q10 = p10 + 2 * plane_stride, *q11 = p11 + 2 * plane_stride;
      const uint32_t ew[4] = {e4.x, e4.y, e4.z, e4.w};
      const int xw0 = sx * K7_SEG;
#pragma unroll
      for (int j = 0; j < K7_SEG; ++j) {
        if ((ew[j >> 2] >> (8 * (j & 3))) & 0xffu) {
          const LinIdx iw = lin_index_ac(xw0 + j, sw, w);
          const float a = id.w0 * (ih.w0 * (iw.w0 * p00[iw.i0] + iw.w1 * p00[iw.i1]) +
                                   ih.w1 * (iw.w0 * p01[iw.i0] + iw.w1 * p01[iw.i1])) +
                          id.w1 * (ih.w0 * (iw.w0 * p10[iw.i0] + iw.w1 * p10[iw.i1]) +
                                   ih.w1 * (iw.w0 * p11[iw.i0] + iw.w1 * p11[iw.i1]));
          const float c = id.w0 * (ih.w0 * (iw.w0 * q00[iw.i0] + iw.w1 * q00[iw.i1]) +
                                   ih.w1 * (iw.w0 * q01[iw.i0] + iw.w1 * q01[iw.i1])) +
                          id.w1 * (ih.w0 * (iw.w0 * q10[iw.i0] + iw.w1 * q10[iw.i1]) +
                                   ih.w1 * (iw.w0 * q11[iw.i0] + iw.w1 * q11[iw.i1]));
          v0[j] = a;
          v1[j] = c;
          acc0 += (double)a;
          acc1 += (double)c;
        }
      }
    }
  }
  // Output: the slice's rows are ONE contiguous run of rows * W floats per map.  It leaves through the bulk-copy engine
  // (cp.async.bulk shared -> global, one instruction per map issued by one thread) instead of per-lane stores: st.global
  // streams topped out near 2 TB/s in this library's write-heavy kernels, TMA stores reach 4.7 (K4).  Slices without an
  // `ess` voxel (~90 % of a chest volume) send the same zeroed 16 KiB tile to both maps.
  {
    float4 *mine0 = reinterpret_cast<float4 *>(stage + threadIdx.x * K7_SEG);
    float4 *mine1 = reinterpret_cast<float4 *>(stage + SLICE + threadIdx.x * K7_SEG);  // thread (sx, ry) = ry * SX + sx
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      mine0[q] = make_float4(v0[4 * q], v0[4 * q + 1], v0[4 * q + 2], v0[4 * q + 3]);
      if (need) mine1[q] = make_float4(v1[4 * q], v1[4 * q + 1], v1[4 * q + 2], v1[4 * q + 3]);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
      const int rows = min(RY, H - xh0);
      const int64_t slice = (int64_t)b * vol + ((int64_t)xd * H + xh0) * W;
      const uint32_t bytes = (uint32_t)rows * (uint32_t)W * 4u;
      const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(stage);
      const uint32_t s1 = need ? s0 + SLICE * 4u : s0;
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out0 + slice), "r"(s0), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out1 + slice), "r"(s1), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
  // lung count: integer warp reductions, one atomic per CTA; map sums only where the CTA met `ess`
  const unsigned wsum = __reduce_add_sync(0xffffffffu, lung_count);
  if ((threadIdx.x & 31) == 0) lung_part[threadIdx.x >> 5] = wsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned tot = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += lung_part[i];
    if (tot) atomicAdd(&sums[2 * n + b], (double)tot);
  }
  if (need) {
    acc0 = block_sum(acc0, scratch);
    if (threadIdx.x == 0) atomicAdd(&sums[b], acc0);
    acc1 = block_sum(acc1, scratch);
    if (threadIdx.x == 0) atomicAdd(&sums[n + b], acc1);
  }
  if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the tiles are read before the CTA leaves
}
__global__ void dram_finalize_kernel(const double *__restrict__ sums, float *__restrict__ pct, int n,
                                     int per_sample) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * n) return;
  const int b = i % n;
  double den = 0.0;
  if (per_sample) den = sums[2 * n + b];
  else
    for (int j = 0; j < n; ++j) den += sums[2 * n + j];
  pct[i] = (float)sums[i] / (float)den;
}

// ---------------------------------------------------------------------------------------
// K7l per-label dRAM sums: for every label k of a uint8 label volume, the voxel count and the sums of both
// dRAM maps over the `ess` voxels labelled k.  Bit-reproducible without floating-point atomics:
//   partial: grid (P, n).  A CTA walks tiles p, p+P, ... of its sample.  Per tile every thread holds 4 x 16
//            labels and ess bytes in registers (16-byte loads, or byte loads on the scalar path), adds its runs of
//            equal labels to shared integer counts and marks the labels that have ess voxels in a 256-bit set;
//            then, for each marked label in increasing order, one fixed-tree block sum (fp64) of the map values
//            (read only at ess voxels) that thread 0 adds to the CTA's accumulator.  Each CTA writes all 256
//            entries of its partial (zeros included).
//   finish:  grid (8, n), 32 labels per CTA; warp w adds partials w, w+8, ... in order, then warps 0..7 in order.
// ---------------------------------------------------------------------------------------
static constexpr int LOBE_THREADS = 256;
static constexpr int LOBE_VECS = 4;                                   // 16-voxel vectors per thread and tile
static constexpr int LOBE_TILE = LOBE_THREADS * LOBE_VECS * 16;       // 16384 voxels
static constexpr int LOBE_LABELS = 256;

__device__ __forceinline__ unsigned byte_of(const uint32_t (&w)[LOBE_VECS * 4], int j, int k) {
  return (w[j * 4 + (k >> 2)] >> (8 * (k & 3))) & 0xffu;
}

template <bool VEC>
__global__ void __launch_bounds__(LOBE_THREADS)
lobe_sums_partial_kernel(const float *__restrict__ map0, const float *__restrict__ map1, const uint8_t *__restrict__ ess,
                         const uint8_t *__restrict__ labels, double *__restrict__ psum, uint32_t *__restrict__ pcnt,
                         int64_t count) {
  __shared__ uint32_t cnt[LOBE_LABELS];
  __shared__ double acc0[LOBE_LABELS], acc1[LOBE_LABELS];
  __shared__ uint32_t marked[LOBE_LABELS / 32];
  __shared__ double2 scratch[32];
  const int t = threadIdx.x, P = gridDim.x;
  const int64_t base = (int64_t)blockIdx.y * count;
  const float *m0 = map0 + base, *m1 = map1 + base;
  const uint8_t *es = ess + base, *lb = labels + base;
  cnt[t] = 0;
  acc0[t] = 0.0;
  acc1[t] = 0.0;
  const int64_t tiles = (count + LOBE_TILE - 1) / LOBE_TILE;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += P) {
    if (t < LOBE_LABELS / 32) marked[t] = 0;
    __syncthreads();
    const int64_t t0 = tile * LOBE_TILE;
    uint32_t lw[LOBE_VECS * 4], ew[LOBE_VECS * 4];
    int nv[LOBE_VECS];
#pragma unroll
    for (int j = 0; j < LOBE_VECS; ++j) {
      const int64_t o = t0 + (int64_t)(j * LOBE_THREADS + t) * 16;
      const int64_t left = count - o;
      nv[j] = left <= 0 ? 0 : (left >= 16 ? 16 : (int)left);
      if constexpr (VEC) {  // count % 16 == 0: a vector is whole or absent
        const uint4 l4 = nv[j] ? __ldg(reinterpret_cast<const uint4 *>(lb + o)) : make_uint4(0, 0, 0, 0);
        const uint4 e4 = nv[j] ? __ldg(reinterpret_cast<const uint4 *>(es + o)) : make_uint4(0, 0, 0, 0);
        lw[j * 4 + 0] = l4.x; lw[j * 4 + 1] = l4.y; lw[j * 4 + 2] = l4.z; lw[j * 4 + 3] = l4.w;
        ew[j * 4 + 0] = e4.x; ew[j * 4 + 1] = e4.y; ew[j * 4 + 2] = e4.z; ew[j * 4 + 3] = e4.w;
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) lw[j * 4 + q] = ew[j * 4 + q] = 0;
        for (int k = 0; k < nv[j]; ++k) {
          lw[j * 4 + (k >> 2)] |= (uint32_t)__ldg(lb + o + k) << (8 * (k & 3));
          ew[j * 4 + (k >> 2)] |= (uint32_t)(__ldg(es + o + k) != 0) << (8 * (k & 3));
        }
      }
    }
    // counts (runs of one label -> one shared atomic), the set of labels with ess voxels, and this thread's map sums
    // over its ess voxels while they carry one label (all map loads of the tile in one burst, before any barrier)
    unsigned cur = LOBE_LABELS, run = 0, last_marked = LOBE_LABELS, mine = LOBE_LABELS;
    double a0 = 0.0, a1 = 0.0;
    bool mixed = false;
#pragma unroll
    for (int j = 0; j < LOBE_VECS; ++j) {
      const int64_t o = t0 + (int64_t)(j * LOBE_THREADS + t) * 16;
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        if (k < nv[j]) {
          const unsigned lab = byte_of(lw, j, k);
          if (lab != cur) {
            if (run) atomicAdd(&cnt[cur], run);
            cur = lab;
            run = 0;
          }
          ++run;
          if (byte_of(ew, j, k)) {
            if (lab != last_marked) {
              atomicOr(&marked[lab >> 5], 1u << (lab & 31));
              last_marked = lab;
            }
            if (mine == LOBE_LABELS) mine = lab;
            if (lab == mine) {
              a0 += (double)__ldg(m0 + o + k);
              a1 += (double)__ldg(m1 + o + k);
            } else {
              mixed = true;
            }
          }
        }
      }
    }
    if (run) atomicAdd(&cnt[cur], run);
    __syncthreads();
    for (int w = 0; w < LOBE_LABELS / 32; ++w) {
      uint32_t set = marked[w];  // the same word in every thread: the loop below is uniform across the CTA
      while (set) {
        const int bit = __ffs(set) - 1;
        set &= set - 1;
        const unsigned label = (unsigned)(w * 32 + bit);
        double s0 = label == mine ? a0 : 0.0, s1 = label == mine ? a1 : 0.0;
        if (mixed) {  // ess voxels of several labels: sum this label's again, in the same voxel order
          s0 = s1 = 0.0;
#pragma unroll
          for (int j = 0; j < LOBE_VECS; ++j) {
            const int64_t o = t0 + (int64_t)(j * LOBE_THREADS + t) * 16;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              if (k < nv[j] && byte_of(ew, j, k) && byte_of(lw, j, k) == label) {
                s0 += (double)__ldg(m0 + o + k);
                s1 += (double)__ldg(m1 + o + k);
              }
            }
          }
        }
        block_sum2(s0, s1, scratch);
        if (t == 0) {
          acc0[label] += s0;
          acc1[label] += s1;
        }
      }
    }
    __syncthreads();  // `marked` is reset for the next tile only after every thread has read it
  }
  __syncthreads();
  const int64_t slot = (int64_t)blockIdx.y * P + blockIdx.x;
  psum[(slot * 2 + 0) * LOBE_LABELS + t] = acc0[t];
  psum[(slot * 2 + 1) * LOBE_LABELS + t] = acc1[t];
  pcnt[slot * LOBE_LABELS + t] = cnt[t];
}

__global__ void __launch_bounds__(256)
lobe_sums_finish_kernel(const double *__restrict__ psum, const uint32_t *__restrict__ pcnt, float *__restrict__ pct,
                        int64_t *__restrict__ voxels, int n, int P) {
  __shared__ double r0[8][32], r1[8][32];
  __shared__ unsigned long long rc[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.y;
  const int label = blockIdx.x * 32 + lane;
  double s0 = 0.0, s1 = 0.0;
  unsigned long long c = 0;
  for (int p = warp; p < P; p += 8) {
    const int64_t slot = (int64_t)b * P + p;
    s0 += psum[(slot * 2 + 0) * LOBE_LABELS + label];
    s1 += psum[(slot * 2 + 1) * LOBE_LABELS + label];
    c += pcnt[slot * LOBE_LABELS + label];
  }
  r0[warp][lane] = s0;
  r1[warp][lane] = s1;
  rc[warp][lane] = c;
  __syncthreads();
  if (warp == 0) {
    for (int w = 1; w < 8; ++w) {
      s0 += r0[w][lane];
      s1 += r1[w][lane];
      c += rc[w][lane];
    }
    const int64_t o = (int64_t)b * LOBE_LABELS + label;
    voxels[o] = (int64_t)c;
    // the conversion of dram_finalize_kernel; 0 / 0 gives NaN for a label without voxels
    pct[o] = (float)s0 / (float)c;
    pct[(int64_t)n * LOBE_LABELS + o] = (float)s1 / (float)c;
  }
}

// ---------------------------------------------------------------------------------------
// K8 HU window + standardise: pass 1 accumulates sum and sum of squares of the windowed
// values in fp64, pass 2 derives mean / unbiased std and writes (v - mean) / std in fp32.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float window_value(short hu, float lo, float hi) {
  float f = (float)hu;
  f = fminf(fmaxf(f, lo), hi);
  return (f - lo) / (hi - lo);
}
// grid = (blocks, n): blockIdx.y = volume.  VEC: 16-byte loads (volumes start 16-byte aligned, count % 8 == 0).
template <bool VEC>
__global__ void __launch_bounds__(256)
window_stats_kernel(const short *__restrict__ hu_all, double *__restrict__ sums_all, int64_t count, float lo, float hi) {
  __shared__ double scratch[32];
  const short *hu = hu_all + (int64_t)blockIdx.y * count;
  double *sums = sums_all + 2 * blockIdx.y;
  double s = 0.0, s2 = 0.0;
  if constexpr (VEC) {
    const int64_t nvec = count / 8;
    const uint4 *hv = reinterpret_cast<const uint4 *>(hu);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // two independent 16-byte loads in flight per thread and iteration
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += 2 * stride) {
      const uint4 u0 = __ldg(hv + i);
      const bool two = i + stride < nvec;
      const uint4 u1 = two ? __ldg(hv + i + stride) : make_uint4(0, 0, 0, 0);
      const uint32_t uu[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
      float ls = 0.0f, ls2 = 0.0f;  // <= 16 values in [0,1]: fp32 is exact enough before widening
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (q >= 4 && !two) break;
        const float a = window_value((short)(uu[q] & 0xffff), lo, hi);
        const float b = window_value((short)(uu[q] >> 16), lo, hi);
        ls += a + b;
        ls2 += a * a + b * b;
      }
      s += (double)ls;
      s2 += (double)ls2;
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
      const float a = window_value(hu[i], lo, hi);
      s += (double)a;
      s2 += (double)(a * a);
    }
  }
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[0], s);
  s2 = block_sum(s2, scratch);
  if (threadIdx.x == 0) atomicAdd(&sums[1], s2);
}
// one thread per volume: stats[v] = (mean, unbiased std); stats_out (optional) gets a copy
__global__ void window_finalize_kernel(const double *__restrict__ sums, float *__restrict__ stats,
                                       float *__restrict__ stats_out, int64_t count, int n) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const double cnt = (double)count;
  const double mean = sums[2 * v] / cnt;
  double var = (sums[2 * v + 1] - cnt * mean * mean) / (cnt - 1.0);
  if (var < 0.0) var = 0.0;
  stats[2 * v] = (float)mean;
  stats[2 * v + 1] = (float)sqrt(var);
  if (stats_out) {
    stats_out[2 * v] = stats[2 * v];
    stats_out[2 * v + 1] = stats[2 * v + 1];
  }
}
// Table of K8's result for every integer HU value of the window: lut[v][i] = ((lo + i - lo) / (hi - lo) - mean_v) / sd_v,
// evaluated with the very expression of window_apply_kernel (clamping is the identity inside the window).
__global__ void window_lut_kernel(const float *__restrict__ stats, float *__restrict__ lut, int size, float lo, float hi) {
  const int v = blockIdx.y;
  const float mean = stats[2 * v], sd = stats[2 * v + 1];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < size; i += gridDim.x * blockDim.x)
    lut[(int64_t)v * size + i] = (window_value((short)((int)lo + i), lo, hi) - mean) / sd;
}
template <bool VEC>
__global__ void __launch_bounds__(256)
window_apply_kernel(const short *__restrict__ hu_all, float *__restrict__ out_all, const float *__restrict__ stats,
                    int64_t count, float lo, float hi) {
  const short *hu = hu_all + (int64_t)blockIdx.y * count;
  float *out = out_all + (int64_t)blockIdx.y * count;
  const float mean = stats[2 * blockIdx.y], sd = stats[2 * blockIdx.y + 1];
  if constexpr (VEC) {
    const int64_t nvec = count / 8;
    const uint4 *hv = reinterpret_cast<const uint4 *>(hu);
    float4 *ov = reinterpret_cast<float4 *>(out);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec;
         i += (int64_t)gridDim.x * blockDim.x) {
      const uint4 u = __ldg(hv + i);
      const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
      float f[8];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        f[2 * q + 0] = (window_value((short)(uu[q] & 0xffff), lo, hi) - mean) / sd;
        f[2 * q + 1] = (window_value((short)(uu[q] >> 16), lo, hi) - mean) / sd;
      }
      ov[2 * i + 0] = make_float4(f[0], f[1], f[2], f[3]);
      ov[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
      out[i] = (window_value(hu[i], lo, hi) - mean) / sd;
  }
}

// ---------------------------------------------------------------------------------------
// K8b Interpolate transform: in-plane bilinear (image) / legacy nearest (mask) + slice pick.
// ---------------------------------------------------------------------------------------
__global__ void resize_image_kernel(const float *__restrict__ x, float *__restrict__ out,
                                    const int *__restrict__ d_idx, int H, int W, int D2, int H2, int W2,
                                    float sh, float sw) {
  const int64_t total = (int64_t)D2 * H2 * W2;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int xw = (int)(t % W2);
    const int64_t r = t / W2;
    const int xh = (int)(r % H2);
    const int xd = (int)(r / H2);
    const float *src = x + (int64_t)__ldg(d_idx + xd) * H * W;
    const LinIdx ih = lin_index_ac(xh, sh, H), iw = lin_index_ac(xw, sw, W);
    const float *r0 = src + (int64_t)ih.i0 * W, *r1 = src + (int64_t)ih.i1 * W;
    out[t] = ih.w0 * (iw.w0 * __ldg(r0 + iw.i0) + iw.w1 * __ldg(r0 + iw.i1)) +
             ih.w1 * (iw.w0 * __ldg(r1 + iw.i0) + iw.w1 * __ldg(r1 + iw.i1));
  }
}
// KEEP = false: the mask rule (0/1 out); KEEP = true: the same voxel picked, its value kept (label volumes).
template <bool KEEP>
__global__ void resize_mask_kernel(const uint8_t *__restrict__ x, uint8_t *__restrict__ out,
                                   const int *__restrict__ d_idx, int H, int W, int D2, int H2, int W2) {
  const int64_t total = (int64_t)D2 * H2 * W2;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int xw = (int)(t % W2);
    const int64_t r = t / W2;
    const int xh = (int)(r % H2);
    const int xd = (int)(r / H2);
    const int zh = nearest_index(xh, H, H2), zw = nearest_index(xw, W, W2);
    const uint8_t v = x[((int64_t)__ldg(d_idx + xd) * H + zh) * W + zw];
    out[t] = KEEP ? v : (v ? 1 : 0);
  }
}

// ---------------------------------------------------------------------------------------
// layout helpers
// ---------------------------------------------------------------------------------------
__global__ void ncdhw_to_ndhwc_kernel(const float *__restrict__ x, uint16_t *__restrict__ out, int n, int c,
                                      int64_t plane, int f16) {
  const int64_t total = (int64_t)n * c * plane;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int ch = (int)(t % c);
    const int64_t v = t / c;  // b*plane + s
    const int64_t b = v / plane, s = v % plane;
    out[t] = store16(x[(b * c + ch) * plane + s], f16);
  }
}
__global__ void ndhwc_to_ncdhw_kernel(const uint16_t *__restrict__ x, float *__restrict__ out, int n, int c,
                                      int64_t plane, int f16) {
  const int64_t total = (int64_t)n * c * plane;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = t % plane;
    const int64_t r = t / plane;  // b*c + ch
    const int64_t b = r / c;
    const int ch = (int)(r % c);
    out[t] = load16(x + (b * plane + s) * c + ch, f16);
  }
}

}  // namespace dram

using namespace dram;

static const int kThreads = 256;

static int dtype_flag(int32_t dtype, int *f16) {
  DRAM_REQUIRE(dtype == DRAM_DTYPE_BF16 || dtype == DRAM_DTYPE_F16, "dtype must be DRAM_DTYPE_BF16 or DRAM_DTYPE_F16");
  *f16 = dtype == DRAM_DTYPE_F16;
  return DRAM_OK;
}

extern "C" int dram_stem_expand(const float *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                                int32_t dtype, void *stream) {
  int f16;
  if (int rc = dtype_flag(dtype, &f16)) return rc;
  DRAM_REQUIRE(x && out, "dram_stem_expand: null pointer");
  DRAM_REQUIRE(n > 0 && d > 0 && h > 0 && w > 0, "dram_stem_expand: empty volume");
  const int h2 = (h - 1) / 2 + 1, w2 = (w - 1) / 2 + 1;
  const int64_t total = (int64_t)n * d * h2 * w2 * 8;
  stem_expand_kernel<<<stream_grid(total, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      x, reinterpret_cast<uint4 *>(out), n, d, h, w, h2, w2, f16);
  DRAM_CHECK_LAUNCH("stem_expand_kernel");
  return DRAM_OK;
}

extern "C" int dram_maxpool3d(const void *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                              int32_t c, int32_t dtype, void *stream) {
  int f16;
  if (int rc = dtype_flag(dtype, &f16)) return rc;
  DRAM_REQUIRE(x && out, "dram_maxpool3d: null pointer");
  DRAM_REQUIRE(n > 0 && d > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0,
               "dram_maxpool3d: bad shape (c must be a multiple of 8)");
  const int od = (d - 1) / 2 + 1, oh = (h - 1) / 2 + 1, ow = (w - 1) / 2 + 1;
  const int dchunks = ceil_div(od, POOL_DCHUNK);
  const int64_t total = (int64_t)n * dchunks * oh * ow * (c / 8);
  DRAM_REQUIRE((int64_t)h * w * (c / 8) < 0x7fffffffLL, "dram_maxpool3d: plane too large");
  const int grid = stream_grid(total, kThreads);
  if (f16)
    maxpool3d_kernel<true><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(x), reinterpret_cast<uint4 *>(out), n, d, h, w, c / 8, od, oh, ow, dchunks);
  else
    maxpool3d_kernel<false><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(x), reinterpret_cast<uint4 *>(out), n, d, h, w, c / 8, od, oh, ow, dchunks);
  DRAM_CHECK_LAUNCH("maxpool3d_kernel");
  return DRAM_OK;
}

extern "C" int dram_upsample2x(const void *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                               int32_t c, int32_t dtype, void *stream) {
  int f16;
  if (int rc = dtype_flag(dtype, &f16)) return rc;
  DRAM_REQUIRE(x && out, "dram_upsample2x: null pointer");
  DRAM_REQUIRE(n > 0 && d > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0,
               "dram_upsample2x: bad shape (c must be a multiple of 8)");
  const int dchunks = ceil_div(2 * d, UP_DCHUNK);
  const int64_t total = (int64_t)n * dchunks * (2 * h) * (2 * w) * (c / 8);
  DRAM_REQUIRE((int64_t)h * w * (c / 8) < 0x7fffffffLL, "dram_upsample2x: plane too large");
  const int grid = stream_grid(total, kThreads);
  if (f16)
    upsample2x_kernel<true><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(x), reinterpret_cast<uint4 *>(out), n, d, h, w, c / 8,
        ac_scale(d, 2 * d), ac_scale(h, 2 * h), ac_scale(w, 2 * w), dchunks);
  else
    upsample2x_kernel<false><<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(x), reinterpret_cast<uint4 *>(out), n, d, h, w, c / 8,
        ac_scale(d, 2 * d), ac_scale(h, 2 * h), ac_scale(w, 2 * w), dchunks);
  DRAM_CHECK_LAUNCH("upsample2x_kernel");
  return DRAM_OK;
}

extern "C" size_t dram_pool_workspace_bytes(int32_t n, int32_t ch) {
  if (n <= 0 || ch <= 0) return 0;
  return sizeof(double) * (size_t)n * (size_t)(ch + 1);
}

extern "C" int dram_masked_pool(const float *dense, const void *mask, int32_t mask_is_f32, float *out,
                                void *workspace, int32_t n, int32_t ch, int32_t d, int32_t h, int32_t w,
                                int32_t md, int32_t mh, int32_t mw, void *stream) {
  DRAM_REQUIRE(dense && out && workspace, "dram_masked_pool: null pointer");
  DRAM_REQUIRE(n > 0 && ch > 0 && ch <= 65535 && d > 0 && h > 0 && w > 0, "dram_masked_pool: bad shape");
  DRAM_REQUIRE(mask == nullptr || (md > 0 && mh > 0 && mw > 0), "dram_masked_pool: bad mask shape");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_cuda(cudaMemsetAsync(workspace, 0, dram_pool_workspace_bytes(n, ch), st),
                      "dram_masked_pool memset");
  if (rc != DRAM_OK) return rc;
  DRAM_REQUIRE((int64_t)d * h < 0x7fffffffLL, "dram_masked_pool: too many rows");
  const bool vec = (w % 4 == 0) && ((uintptr_t)dense % 16 == 0);
  int blocks = stream_grid((int64_t)d * h * 32, kThreads, 8);  // one warp per row
  int per = blocks / (n * ch);
  if (per < 1) per = 1;
  dim3 grid(per, ch, n);
  double *ws = reinterpret_cast<double *>(workspace);
  if (mask_is_f32) {
    const float *mf = reinterpret_cast<const float *>(mask);
    if (vec) masked_pool_partial_kernel<float, 4><<<grid, kThreads, 0, st>>>(dense, mf, ws, ch, d, h, w, md, mh, mw);
    else masked_pool_partial_kernel<float, 1><<<grid, kThreads, 0, st>>>(dense, mf, ws, ch, d, h, w, md, mh, mw);
  } else {
    const uint8_t *mu = reinterpret_cast<const uint8_t *>(mask);
    if (vec) masked_pool_partial_kernel<uint8_t, 4><<<grid, kThreads, 0, st>>>(dense, mu, ws, ch, d, h, w, md, mh, mw);
    else masked_pool_partial_kernel<uint8_t, 1><<<grid, kThreads, 0, st>>>(dense, mu, ws, ch, d, h, w, md, mh, mw);
  }
  DRAM_CHECK_LAUNCH("masked_pool_partial_kernel");
  masked_pool_finalize_kernel<<<ceil_div(n * ch, 128), 128, 0, st>>>(
      reinterpret_cast<const double *>(workspace), out, n, ch);
  DRAM_CHECK_LAUNCH("masked_pool_finalize_kernel");
  return DRAM_OK;
}

extern "C" size_t dram_dram_workspace_bytes(int32_t n) {
  if (n <= 0) return 0;
  return sizeof(double) * 3 * (size_t)n;
}

extern "C" int dram_dram_upsample_mask(const float *dense0, const float *dense1, const uint8_t *ess,
                                       const uint8_t *lungs, float *out0, float *out1, float *pct,
                                       void *workspace, int32_t n, int32_t d, int32_t h, int32_t w,
                                       int32_t D, int32_t H, int32_t W, int32_t per_sample_denominator,
                                       void *stream) {
  DRAM_REQUIRE(dense0 && dense1 && ess && lungs && out0 && out1 && pct && workspace,
               "dram_dram_upsample_mask: null pointer");
  DRAM_REQUIRE(n > 0 && d > 0 && h > 0 && w > 0 && D > 0 && H > 0 && W > 0,
               "dram_dram_upsample_mask: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_cuda(cudaMemsetAsync(workspace, 0, dram_dram_workspace_bytes(n), st),
                      "dram_dram_upsample_mask memset");
  if (rc != DRAM_OK) return rc;
  const float sd = ac_scale(d, D), sh = ac_scale(h, H), sw = ac_scale(w, W);
  DRAM_REQUIRE((int64_t)D * H < 0x7fffffffLL && (int64_t)d * h * w < 0x7fffffffLL,
               "dram_dram_upsample_mask: volume too large for 32-bit row indices");
  double *sums = reinterpret_cast<double *>(workspace);
  // Staged kernel: RH rows per CTA so that RH * ceil(W/16) segments keep 256 threads busy (at most two per thread);
  // the brick of source rows they read is at most nr_max = ceil(RH * (h-1)/(H-1)) + 2 rows per plane.
  const int segs = ceil_div(W, K7_SEG);
  int RH = 1;
  while (RH < 32 && 2 * RH * segs <= 2 * K7_THREADS) RH *= 2;
  const char *k7_env = getenv("DRAM_B200_K7");
  const bool staged_ok = RH * segs <= 2 * K7_THREADS && !(k7_env && strcmp(k7_env, "rows") == 0);
  const int nr_max = (int)ceilf((float)RH * sh) + 2 < h ? (int)ceilf((float)RH * sh) + 2 : h;
  const size_t smem = (size_t)4 * nr_max * w * sizeof(float);
  // lean kernel: W = 16 * 2^k segments per row (k = 2..6), one CTA per RY-row slice of a plane
  int log_sx = -1;
  for (int k = 2; k <= 6; ++k)
    if (W == (K7_SEG << k)) log_sx = k;
  const bool aligned16 = (w % 4 == 0) && (((uintptr_t)ess | (uintptr_t)lungs) % 16 == 0) &&
                         (((uintptr_t)out0 | (uintptr_t)out1 | (uintptr_t)dense0 | (uintptr_t)dense1) % 16 == 0) &&
                         (((int64_t)D * H * W) % 16 == 0) && (((int64_t)d * h * w) % 4 == 0);
  const bool lean_env = !(k7_env && (strcmp(k7_env, "rows") == 0 || strcmp(k7_env, "staged") == 0));
  if (lean_env && log_sx >= 0 && aligned16 && D <= 65535 && n <= 65535) {
    const int RY = 256 >> log_sx;
    const int nr_lean = (int)ceilf((float)RY * sh) + 2 < h ? (int)ceilf((float)RY * sh) + 2 : h;
    const size_t smem_lean = (size_t)(2 * 256 * K7_SEG + 4 * nr_lean * w) * sizeof(float);  // 2 output tiles + the brick
    if (smem_lean <= 160 * 1024) {
      dim3 grid(ceil_div(H, RY), D, n);
#define DRAM_K7_LEAN(LS)                                                                                                  \
  do {                                                                                                                    \
    rc = check_cuda(cudaFuncSetAttribute(dram_upsample_mask_lean_kernel<LS>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         (int)smem_lean),                                                                 \
                    "cudaFuncSetAttribute(dram_upsample_mask_lean_kernel)");                                              \
    if (rc != DRAM_OK) return rc;                                                                                         \
    dram_upsample_mask_lean_kernel<LS><<<grid, 256, smem_lean, st>>>(dense0, dense1, ess, lungs, out0, out1, sums, n, d,  \
                                                                     h, w, D, H, W, sd, sh, sw, nr_lean);                 \
  } while (0)
      switch (log_sx) {
        case 2: DRAM_K7_LEAN(2); break;
        case 3: DRAM_K7_LEAN(3); break;
        case 4: DRAM_K7_LEAN(4); break;
        case 5: DRAM_K7_LEAN(5); break;
        default: DRAM_K7_LEAN(6); break;
      }
#undef DRAM_K7_LEAN
      DRAM_CHECK_LAUNCH("dram_upsample_mask_lean_kernel");
      dram_finalize_kernel<<<ceil_div(2 * n, 128), 128, 0, st>>>(sums, pct, n, per_sample_denominator);
      DRAM_CHECK_LAUNCH("dram_finalize_kernel");
      return DRAM_OK;
    }
  }
  if (staged_ok && smem <= 160 * 1024) {
    const bool fast = (W % 16 == 0) && (w % 4 == 0) && (((uintptr_t)ess | (uintptr_t)lungs) % 16 == 0) &&
                      (((uintptr_t)out0 | (uintptr_t)out1 | (uintptr_t)dense0 | (uintptr_t)dense1) % 16 == 0) &&
                      (((int64_t)D * H * W) % 16 == 0) && (((int64_t)d * h * w) % 4 == 0);
    const int groups = D * ceil_div(H, RH);
    int per = (sm_count() * 6) / n;
    if (per < 1) per = 1;
    if (per > groups) per = groups;
    dim3 grid(per, n);
    if (fast) {
      rc = check_cuda(cudaFuncSetAttribute(dram_upsample_mask_staged_kernel<true>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                      "cudaFuncSetAttribute(dram_upsample_mask_staged_kernel)");
      if (rc != DRAM_OK) return rc;
      dram_upsample_mask_staged_kernel<true><<<grid, K7_THREADS, smem, st>>>(dense0, dense1, ess, lungs, out0, out1, sums, n,
                                                                            d, h, w, D, H, W, sd, sh, sw, RH, nr_max);
    } else {
      rc = check_cuda(cudaFuncSetAttribute(dram_upsample_mask_staged_kernel<false>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                      "cudaFuncSetAttribute(dram_upsample_mask_staged_kernel)");
      if (rc != DRAM_OK) return rc;
      dram_upsample_mask_staged_kernel<false><<<grid, K7_THREADS, smem, st>>>(dense0, dense1, ess, lungs, out0, out1, sums,
                                                                             n, d, h, w, D, H, W, sd, sh, sw, RH, nr_max);
    }
    DRAM_CHECK_LAUNCH("dram_upsample_mask_staged_kernel");
  } else {
    const bool vec = (W % 4 == 0) && (((uintptr_t)ess | (uintptr_t)lungs) % 4 == 0) &&
                     (((uintptr_t)out0 | (uintptr_t)out1) % 16 == 0);
    int bps = stream_grid((int64_t)D * H * 32, kThreads, 8) / n;  // one warp per output row
    if (bps < 1) bps = 1;
    if (vec)
      dram_upsample_mask_kernel<4><<<bps * n, kThreads, 0, st>>>(dense0, dense1, ess, lungs, out0, out1, sums,
                                                                 n, d, h, w, D, H, W, sd, sh, sw, bps);
    else
      dram_upsample_mask_kernel<1><<<bps * n, kThreads, 0, st>>>(dense0, dense1, ess, lungs, out0, out1, sums,
                                                                 n, d, h, w, D, H, W, sd, sh, sw, bps);
    DRAM_CHECK_LAUNCH("dram_upsample_mask_kernel");
  }
  dram_finalize_kernel<<<ceil_div(2 * n, 128), 128, 0, st>>>(sums, pct, n, per_sample_denominator);
  DRAM_CHECK_LAUNCH("dram_finalize_kernel");
  return DRAM_OK;
}

// CTAs per sample of the per-label sums: ~1024 in all, at least two tiles each.  A function of the shape only, so the
// summation order (and with it every bit of the result) does not depend on the device.
static int lobe_ctas(int32_t n, int64_t count) {
  const int64_t tiles = ceil_div64(count, LOBE_TILE);
  int64_t p = ceil_div64(tiles, 2);
  const int64_t cap = n >= 1024 ? 1 : 1024 / n;
  if (p > cap) p = cap;
  return p < 1 ? 1 : (int)p;
}

extern "C" size_t dram_lobe_workspace_bytes(int32_t n, int64_t count) {
  if (n <= 0 || count <= 0) return 0;
  return (size_t)n * lobe_ctas(n, count) * LOBE_LABELS * (2 * sizeof(double) + sizeof(uint32_t));
}

extern "C" int dram_lobe_sums(const float *map0, const float *map1, const uint8_t *ess, const uint8_t *labels,
                              float *pct, int64_t *voxels, void *workspace, int32_t n, int64_t count, void *stream) {
  DRAM_REQUIRE(map0 && map1 && ess && labels && pct && voxels && workspace, "dram_lobe_sums: null pointer");
  DRAM_REQUIRE(n > 0 && n <= 65535 && count > 0, "dram_lobe_sums: bad shape");
  DRAM_REQUIRE(count < 0x7fffffffLL, "dram_lobe_sums: volume too large for 32-bit per-CTA counts");
  DRAM_REQUIRE((uintptr_t)workspace % 8 == 0, "dram_lobe_sums: workspace must be 8-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int P = lobe_ctas(n, count);
  double *psum = reinterpret_cast<double *>(workspace);
  uint32_t *pcnt = reinterpret_cast<uint32_t *>(psum + (size_t)n * P * 2 * LOBE_LABELS);
  const bool vec = (count % 16 == 0) && (((uintptr_t)ess | (uintptr_t)labels) % 16 == 0);
  dim3 grid(P, n);
  if (vec) lobe_sums_partial_kernel<true><<<grid, LOBE_THREADS, 0, st>>>(map0, map1, ess, labels, psum, pcnt, count);
  else lobe_sums_partial_kernel<false><<<grid, LOBE_THREADS, 0, st>>>(map0, map1, ess, labels, psum, pcnt, count);
  DRAM_CHECK_LAUNCH("lobe_sums_partial_kernel");
  lobe_sums_finish_kernel<<<dim3(LOBE_LABELS / 32, n), 256, 0, st>>>(psum, pcnt, pct, voxels, n, P);
  DRAM_CHECK_LAUNCH("lobe_sums_finish_kernel");
  return DRAM_OK;
}

extern "C" size_t dram_preprocess_workspace_bytes(void) { return 2 * sizeof(double) + 2 * sizeof(float); }
extern "C" size_t dram_preprocess_workspace_bytes_n(int32_t n) {
  return n > 0 ? (size_t)n * (2 * sizeof(double) + 2 * sizeof(float)) : 0;
}

// memset + statistics of all n volumes in one launch + finalize; leaves (mean, std) per volume at workspace + 16 n.
static int window_stats_launch(const int16_t *hu, float *stats_out, void *workspace, int32_t n, int64_t count, float lo,
                               float hi, cudaStream_t st, bool *vec_out) {
  DRAM_REQUIRE(hu && workspace, "dram_window_stats: null pointer");
  DRAM_REQUIRE(n > 0 && n <= 65535, "dram_window_stats: bad volume count");
  DRAM_REQUIRE(count > 1, "dram_window_stats: need at least 2 voxels for an unbiased std");
  DRAM_REQUIRE(hi > lo, "dram_window_stats: empty window");
  DRAM_REQUIRE((uintptr_t)workspace % 8 == 0, "dram_window_stats: workspace must be 8-byte aligned");
  double *sums = reinterpret_cast<double *>(workspace);
  float *stats = reinterpret_cast<float *>(sums + 2 * n);
  int rc = check_cuda(cudaMemsetAsync(workspace, 0, 2 * sizeof(double) * (size_t)n, st), "dram_window_stats memset");
  if (rc != DRAM_OK) return rc;
  // 16-byte loads need every volume to start on a 16-byte boundary
  const bool vec = ((uintptr_t)hu % 16 == 0) && (count % 8 == 0);
  int per = stream_grid(count / 16 + 1, kThreads, 8) / n;
  if (per < 1) per = 1;
  dim3 grid(per, n);
  if (vec) window_stats_kernel<true><<<grid, kThreads, 0, st>>>(hu, sums, count, lo, hi);
  else window_stats_kernel<false><<<grid, kThreads, 0, st>>>(hu, sums, count, lo, hi);
  DRAM_CHECK_LAUNCH("window_stats_kernel");
  window_finalize_kernel<<<ceil_div(n, 64), 64, 0, st>>>(sums, stats, stats_out, count, n);
  DRAM_CHECK_LAUNCH("window_finalize_kernel");
  if (vec_out) *vec_out = vec;
  return DRAM_OK;
}

extern "C" int dram_window_stats(const int16_t *hu, float *stats_out, void *workspace, int32_t n, int64_t count,
                                 float lo, float hi, void *stream) {
  DRAM_REQUIRE(stats_out, "dram_window_stats: stats_out is required");
  return window_stats_launch(hu, stats_out, workspace, n, count, lo, hi, (cudaStream_t)stream, nullptr);
}

extern "C" int dram_window_lut(const int16_t *hu, float *lut, float *stats_out, void *workspace, int32_t n,
                               int64_t count, float lo, float hi, void *stream) {
  DRAM_REQUIRE(lut, "dram_window_lut: lut is required");
  DRAM_REQUIRE(lo == floorf(lo) && hi == floorf(hi) && lo >= -32768.0f && hi <= 32767.0f &&
                   (int)hi - (int)lo + 1 <= DRAM_WINDOW_LUT_MAX,
               "dram_window_lut: the window must have integral bounds inside int16 and at most %d values",
               DRAM_WINDOW_LUT_MAX);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = window_stats_launch(hu, stats_out, workspace, n, count, lo, hi, st, nullptr);
  if (rc != DRAM_OK) return rc;
  const float *stats = reinterpret_cast<const float *>(reinterpret_cast<double *>(workspace) + 2 * n);
  const int size = (int)hi - (int)lo + 1;
  window_lut_kernel<<<dim3(ceil_div(size, 256), n), 256, 0, st>>>(stats, lut, size, lo, hi);
  DRAM_CHECK_LAUNCH("window_lut_kernel");
  return DRAM_OK;
}

extern "C" int dram_window_standardize_batch(const int16_t *hu, float *out, float *stats_out, void *workspace,
                                             int32_t n, int64_t count, float lo, float hi, void *stream) {
  DRAM_REQUIRE(out, "dram_window_standardize: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  bool vec = false;
  int rc = window_stats_launch(hu, stats_out, workspace, n, count, lo, hi, st, &vec);
  if (rc != DRAM_OK) return rc;
  vec = vec && ((uintptr_t)out % 16 == 0);
  const float *stats = reinterpret_cast<const float *>(reinterpret_cast<double *>(workspace) + 2 * n);
  int per = stream_grid(count / 8 + 1, kThreads, 8) / n;
  if (per < 1) per = 1;
  dim3 grid(per, n);
  if (vec) window_apply_kernel<true><<<grid, kThreads, 0, st>>>(hu, out, stats, count, lo, hi);
  else window_apply_kernel<false><<<grid, kThreads, 0, st>>>(hu, out, stats, count, lo, hi);
  DRAM_CHECK_LAUNCH("window_apply_kernel");
  return DRAM_OK;
}

extern "C" int dram_window_standardize(const int16_t *hu, float *out, float *stats_out, void *workspace,
                                       int64_t count, float lo, float hi, void *stream) {
  return dram_window_standardize_batch(hu, out, stats_out, workspace, 1, count, lo, hi, stream);
}

extern "C" int dram_resize_image(const float *x, float *out, const int32_t *d_idx, int32_t D, int32_t H,
                                 int32_t W, int32_t D2, int32_t H2, int32_t W2, void *stream) {
  DRAM_REQUIRE(x && out && d_idx, "dram_resize_image: null pointer");
  DRAM_REQUIRE(D > 0 && H > 0 && W > 0 && D2 > 0 && H2 > 0 && W2 > 0, "dram_resize_image: bad shape");
  const int64_t total = (int64_t)D2 * H2 * W2;
  resize_image_kernel<<<stream_grid(total, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      x, out, d_idx, H, W, D2, H2, W2, ac_scale(H, H2), ac_scale(W, W2));
  DRAM_CHECK_LAUNCH("resize_image_kernel");
  return DRAM_OK;
}

extern "C" int dram_resize_mask(const uint8_t *x, uint8_t *out, const int32_t *d_idx, int32_t D, int32_t H,
                                int32_t W, int32_t D2, int32_t H2, int32_t W2, void *stream) {
  DRAM_REQUIRE(x && out && d_idx, "dram_resize_mask: null pointer");
  DRAM_REQUIRE(D > 0 && H > 0 && W > 0 && D2 > 0 && H2 > 0 && W2 > 0, "dram_resize_mask: bad shape");
  const int64_t total = (int64_t)D2 * H2 * W2;
  resize_mask_kernel<false><<<stream_grid(total, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      x, out, d_idx, H, W, D2, H2, W2);
  DRAM_CHECK_LAUNCH("resize_mask_kernel");
  return DRAM_OK;
}

extern "C" int dram_resize_labels(const uint8_t *x, uint8_t *out, const int32_t *d_idx, int32_t D, int32_t H,
                                  int32_t W, int32_t D2, int32_t H2, int32_t W2, void *stream) {
  DRAM_REQUIRE(x && out && d_idx, "dram_resize_labels: null pointer");
  DRAM_REQUIRE(D > 0 && H > 0 && W > 0 && D2 > 0 && H2 > 0 && W2 > 0, "dram_resize_labels: bad shape");
  const int64_t total = (int64_t)D2 * H2 * W2;
  resize_mask_kernel<true><<<stream_grid(total, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      x, out, d_idx, H, W, D2, H2, W2);
  DRAM_CHECK_LAUNCH("resize_labels_kernel");
  return DRAM_OK;
}

extern "C" int dram_ncdhw_f32_to_ndhwc_16(const float *x, void *out, int32_t n, int32_t c, int32_t d,
                                          int32_t h, int32_t w, int32_t dtype, void *stream) {
  int f16;
  if (int rc = dtype_flag(dtype, &f16)) return rc;
  DRAM_REQUIRE(x && out && n > 0 && c > 0 && d > 0 && h > 0 && w > 0, "dram_ncdhw_f32_to_ndhwc_16: bad argument");
  const int64_t plane = (int64_t)d * h * w;
  ncdhw_to_ndhwc_kernel<<<stream_grid(plane * n * c, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      x, reinterpret_cast<uint16_t *>(out), n, c, plane, f16);
  DRAM_CHECK_LAUNCH("ncdhw_to_ndhwc_kernel");
  return DRAM_OK;
}

extern "C" int dram_ndhwc_16_to_ncdhw_f32(const void *x, float *out, int32_t n, int32_t c, int32_t d,
                                          int32_t h, int32_t w, int32_t dtype, void *stream) {
  int f16;
  if (int rc = dtype_flag(dtype, &f16)) return rc;
  DRAM_REQUIRE(x && out && n > 0 && c > 0 && d > 0 && h > 0 && w > 0, "dram_ndhwc_16_to_ncdhw_f32: bad argument");
  const int64_t plane = (int64_t)d * h * w;
  ndhwc_to_ncdhw_kernel<<<stream_grid(plane * n * c, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint16_t *>(x), out, n, c, plane, f16);
  DRAM_CHECK_LAUNCH("ndhwc_to_ncdhw_kernel");
  return DRAM_OK;
}
