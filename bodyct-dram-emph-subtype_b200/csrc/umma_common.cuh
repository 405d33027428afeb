// Shared device code of the tcgen05 convolution kernels: PTX wrappers (mbarrier, TMA, tcgen05) and the
// fused epilogue (scale/shift, residual incl. shortcut type A, ReLU, 16-bit NDHWC store, 1x1x1 heads).
#pragma once
#include <cuda.h>

#include "common.h"

namespace dram {

// Epilogue description shared by every conv kernel variant.
struct EpiParams {
  int Do, Ho, Wo;              // output spatial dims
  int cout;
  int relu;
  int is_f16;                  // operand/activation storage: 0 = bf16, 1 = fp16 (same 2-byte layout)
  const float *bias;
  const float *scale;          // optional fp32 per-channel multiplier applied to the accumulator
  uint16_t *out;
  const uint16_t *res;
  int res_c, res_stride, res_d, res_h, res_w;
  int n_heads, head_ch0, head_ch1, head_sigmoid, store_out;
  const float *head_w;
  const float *head_b;
  float *head_out0;
  float *head_out1;
  // fp16 storage only: when non-null, every epilogue group whose result exceeds the finite fp16 range (and is
  // clamped to +-65504 by the saturating conversion) adds one to this device counter (dram_set_saturation_counter)
  unsigned int *sat_count;
};

// The calling thread's saturation counter (capi.cu); the conv launchers copy it into the kernel parameters.
unsigned int *current_sat_counter();
inline EpiParams with_sat_counter(EpiParams e) {
  e.sat_count = e.is_f16 ? current_sat_counter() : nullptr;
  return e;
}

// ----------------------------------------------------------------------------------------
// PTX wrappers
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// One lane of a converged warp; the surrounding control flow stays warp-uniform so ptxas keeps
// descriptors and addresses in uniform registers (no R2UR / waterfall loop per tcgen05.mma).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// Warp index that ptxas can prove warp-uniform (shuffle broadcast from lane 0).
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Waits for the phase with the given parity.  A wait longer than ~4 s of SM clocks is a
// protocol bug: trap instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    long long now = clock64();
    if (t0 == 0) t0 = now;
    else if (now - t0 > 8000000000LL) {
      printf("dram_b200: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n",
             blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap *map, uint32_t bar,
                                            int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// smem -> global tile store (bulk async group); the tensor map clips rows outside the tensor.
__device__ __forceinline__ void tma_store_5d(const CUtensorMap *map, uint32_t src, int c0, int c1, int c2, int c3,
                                             int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
      ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap *map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, issued by one thread for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on the mbarrier once every tcgen05.mma issued so far by this thread has retired.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4, [16,30) LBO>>4 (unused for swizzled K-major), [32,46) SBO>>4 = 8 rows * 128 B,
// [46,48) version = 1, [61,64) layout = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// cute::UMMA::InstrDescriptor: c_format F32 (1<<4), a/b format (0 = F16, 1 = BF16) at bits 7 and
// 10, K-major A and B, n_dim = N>>3 at bit 17, m_dim = M>>4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc_16bit(int m, int n, int is_f16) {
  return (1u << 4) | ((is_f16 ? 0u : 1u) << 7) | ((is_f16 ? 0u : 1u) << 10) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// Two packed 16-bit activations <-> fp32, for either storage type.
__device__ __forceinline__ float2 unpack2(uint32_t u, int is_f16) {
  if (is_f16) return __half22float2(*reinterpret_cast<const __half2 *>(&u));
  const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162 *>(&u);
  return make_float2(__low2float(h), __high2float(h));
}
__device__ __forceinline__ uint32_t pack2(float a, float b, int is_f16) {
  if (is_f16) {
    // one F2FP.SATFINITE: values beyond +-65504 saturate instead of overflowing to inf
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t *>(&h);
}


// Saturation probe (debug / first-run check): one atomic per 32-value group that left the fp16 range.  The branch on
// e.sat_count is uniform over the grid, so the default (nullptr) costs one predicate per group.
__device__ __forceinline__ void note_saturation(const EpiParams &e, const float (&y)[32]) {
  float m = 0.0f;
#pragma unroll
  for (int j = 0; j < 32; ++j) m = fmaxf(m, fabsf(y[j]));
  if (!(m <= 65504.0f)) atomicAdd(e.sat_count, 1u);  // also catches NaN
}
// ReLU folded into the conversion (cvt ... .relu clamps negative results to zero): saves one FMNMX per value in the
// epilogues, which matter for the instruction-issue-bound kernels (stem, 1x1x1 convolutions).
__device__ __forceinline__ uint32_t pack2_relu(float a, float b, int is_f16) {
  uint32_t r;
  if (is_f16) asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  else asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

// Residual row of an output voxel (nullptr when there is no residual or the voxel is out of range).
__device__ __forceinline__ const uint16_t *residual_row(const EpiParams &e, bool valid, int sample, int od,
                                                        int oh, int ow) {
  if (e.res == nullptr || !valid) return nullptr;
  const size_t rvox = (((size_t)sample * e.res_d + (size_t)od * e.res_stride) * e.res_h +
                       (size_t)oh * e.res_stride) * e.res_w + (size_t)ow * e.res_stride;
  return e.res + rvox * e.res_c;
}

// The 64 residual bytes of one 32-channel group of a voxel, loaded EARLY: the epilogue loops issue these loads for the
// next group before they wait for the current group's accumulator (tcgen05.ld) and do its arithmetic, so the L2 / DRAM
// latency of the residual row (a different 128-byte line per lane) overlaps work instead of preceding it — the
// convolutions with a residual ran 3 % (tile kernel) to 25 % (plane ring, 64 channels) slower than their twins without.
struct ResGroup {
  uint4 r[4];
  bool on;
};
__device__ __forceinline__ ResGroup load_residual_group(const EpiParams &e, const uint16_t *res_row, int cg) {
  ResGroup g;
  g.on = res_row != nullptr && cg < e.res_c;
  if (g.on) {
    const uint4 *r4 = reinterpret_cast<const uint4 *>(res_row + cg);
#pragma unroll
    for (int j = 0; j < 4; ++j) g.r[j] = __ldg(r4 + j);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) g.r[j] = make_uint4(0u, 0u, 0u, 0u);
  }
  return g;
}

// One 32-column group of one accumulator row: v = raw fp32 accumulator bits, cg = first global output
// channel of the group, res = the group's residual values (load_residual_group).  HEADS: evaluate the fused 1x1x1
// heads (only meaningful when cout == 32).
template <bool HEADS>
__device__ __forceinline__ void epilogue_group(const EpiParams &e, const uint32_t (&v)[32], int cg, int sample,
                                               int od, int oh, int ow, const ResGroup &res) {
  float y[32];
  const float4 *b4 = reinterpret_cast<const float4 *>(e.bias + cg);
  if (e.scale != nullptr) {
    const float4 *s4 = reinterpret_cast<const float4 *>(e.scale + cg);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j), sc = __ldg(s4 + j);
      y[4 * j + 0] = fmaf(__uint_as_float(v[4 * j + 0]), sc.x, b.x);
      y[4 * j + 1] = fmaf(__uint_as_float(v[4 * j + 1]), sc.y, b.y);
      y[4 * j + 2] = fmaf(__uint_as_float(v[4 * j + 2]), sc.z, b.z);
      y[4 * j + 3] = fmaf(__uint_as_float(v[4 * j + 3]), sc.w, b.w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j);
      y[4 * j + 0] = __uint_as_float(v[4 * j + 0]) + b.x;
      y[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
      y[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
      y[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
    }
  }
  if (res.on) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 r = res.r[j];
      const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 f = unpack2(w[q], e.is_f16);
        y[8 * j + 2 * q + 0] += f.x;
        y[8 * j + 2 * q + 1] += f.y;
      }
    }
  }
  // the fp32 ReLU is only needed by the heads and the saturation probe; otherwise the conversion does it
  const bool relu_in_cvt = e.relu && !(HEADS && e.n_heads > 0) && e.sat_count == nullptr;
  if (e.relu && !relu_in_cvt) {
#pragma unroll
    for (int j = 0; j < 32; ++j) y[j] = fmaxf(y[j], 0.0f);
  }
  if (e.sat_count != nullptr && e.store_out) note_saturation(e, y);
  const size_t vox = (((size_t)sample * e.Do + od) * e.Ho + oh) * e.Wo + ow;
  if (e.store_out) {
    uint4 *o4 = reinterpret_cast<uint4 *>(e.out + vox * e.cout + cg);
    if (relu_in_cvt) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] = pack2_relu(y[8 * j + 2 * q], y[8 * j + 2 * q + 1], e.is_f16);
        o4[j] = make_uint4(w[0], w[1], w[2], w[3]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] = pack2(y[8 * j + 2 * q], y[8 * j + 2 * q + 1], e.is_f16);
        o4[j] = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
  }
  if (HEADS && e.n_heads > 0) {
    // 1x1x1 heads on the fp32 post-ReLU vector; dense maps are fp32 NCDHW.
    const size_t plane = (size_t)e.Do * e.Ho * e.Wo;
    const size_t sp = ((size_t)od * e.Ho + oh) * e.Wo + ow;
    const int total = e.head_ch0 + e.head_ch1;
    for (int hc = 0; hc < total; ++hc) {
      const float4 *w4 = reinterpret_cast<const float4 *>(e.head_w + hc * 32);
      float s = __ldg(e.head_b + hc);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 w = __ldg(w4 + j);
        s = fmaf(w.x, y[4 * j + 0], s);
        s = fmaf(w.y, y[4 * j + 1], s);
        s = fmaf(w.z, y[4 * j + 2], s);
        s = fmaf(w.w, y[4 * j + 3], s);
      }
      if (e.head_sigmoid) s = 1.0f / (1.0f + expf(-s));
      if (hc < e.head_ch0)
        e.head_out0[((size_t)sample * e.head_ch0 + hc) * plane + sp] = s;
      else
        e.head_out1[((size_t)sample * e.head_ch1 + (hc - e.head_ch0)) * plane + sp] = s;
    }
  }
}

// Staged variant of one 32-column group: residual row from a SWIZZLE_128B shared-memory tile (or none), result
// written to a SWIZZLE_128B shared-memory tile that a TMA store sends out.  `row` = tile row, `half` = which 64-byte
// half of the 128-byte row this group occupies (0 / 1), cg = first global output channel (for scale / bias).
__device__ __forceinline__ void epilogue_group_staged(const EpiParams &e, const uint32_t (&v)[32], int cg, int row,
                                                      int half, uint32_t res_tile, bool has_res, uint32_t out_tile) {
  float y[32];
  const float4 *b4 = reinterpret_cast<const float4 *>(e.bias + cg);
  if (e.scale != nullptr) {
    const float4 *s4 = reinterpret_cast<const float4 *>(e.scale + cg);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j), sc = __ldg(s4 + j);
      y[4 * j + 0] = fmaf(__uint_as_float(v[4 * j + 0]), sc.x, b.x);
      y[4 * j + 1] = fmaf(__uint_as_float(v[4 * j + 1]), sc.y, b.y);
      y[4 * j + 2] = fmaf(__uint_as_float(v[4 * j + 2]), sc.z, b.z);
      y[4 * j + 3] = fmaf(__uint_as_float(v[4 * j + 3]), sc.w, b.w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j);
      y[4 * j + 0] = __uint_as_float(v[4 * j + 0]) + b.x;
      y[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
      y[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
      y[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
    }
  }
  const uint32_t row_off = (uint32_t)row * 128u;
  if (has_res) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t chunk = (uint32_t)(((half * 4 + j) ^ (row & 7)) << 4);
      uint32_t w[4];
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3])
                   : "r"(res_tile + row_off + chunk));
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 f = unpack2(w[q], e.is_f16);
        y[8 * j + 2 * q + 0] += f.x;
        y[8 * j + 2 * q + 1] += f.y;
      }
    }
  }
  const bool relu_in_cvt = e.relu && e.sat_count == nullptr;
  if (e.relu && !relu_in_cvt) {
#pragma unroll
    for (int j = 0; j < 32; ++j) y[j] = fmaxf(y[j], 0.0f);
  }
  if (e.sat_count != nullptr) note_saturation(e, y);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      w[q] = relu_in_cvt ? pack2_relu(y[8 * j + 2 * q], y[8 * j + 2 * q + 1], e.is_f16)
                         : pack2(y[8 * j + 2 * q], y[8 * j + 2 * q + 1], e.is_f16);
    const uint32_t chunk = (uint32_t)(((half * 4 + j) ^ (row & 7)) << 4);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(out_tile + row_off + chunk), "r"(w[0]), "r"(w[1]),
                 "r"(w[2]), "r"(w[3])
                 : "memory");
  }
}

// Host helpers shared by the plan builders (conv3d_umma.cu).
int encode_act_map(CUtensorMap *map, const void *base, int n, int d, int h, int w, int c, int box_c, int bw,
                   int bh, int bd, int sw, int sh, int sd, int is_f16, int bn = 1);
int encode_weight_map(CUtensorMap *map, const void *base, int cout, int64_t ktot, int block_n, int is_f16);

}  // namespace dram
