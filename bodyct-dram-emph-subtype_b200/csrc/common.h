// Shared host/device helpers for libdram_b200.so (internal; the public ABI is include/dram_b200.h).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "dram_b200.h"

namespace dram {

// Per-thread error text behind dram_last_error().
void set_error(const char *fmt, ...);

inline int check_cuda(cudaError_t e, const char *what) {
  if (e == cudaSuccess) return DRAM_OK;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return DRAM_E_LAUNCH;
}

#define DRAM_REQUIRE(cond, ...)       \
  do {                                \
    if (!(cond)) {                    \
      ::dram::set_error(__VA_ARGS__); \
      return DRAM_E_ARG;              \
    }                                 \
  } while (0)

#define DRAM_CHECK_LAUNCH(what)                                       \
  do {                                                                \
    int _rc = ::dram::check_cuda(cudaGetLastError(), what);           \
    if (_rc != DRAM_OK) return _rc;                                   \
  } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// decoder_mask.cu: the ascending list (and count) of the `total` items of a kernel whose tw x th x td output box, grown
// by `radius` voxels, meets the support bit mask `bits` [n][d][h][ceil(w/32)] (dram_decoder_support).  Items are
// numbered with D fastest (d_fastest) or W fastest; `flags` is scratch of `total` bytes.
int worklist_build(const uint32_t *bits, int n, int d, int h, int w, int tw, int th, int td, int d_fastest, int radius,
                   uint8_t *flags, int *list, int *count, int total, cudaStream_t st);

// Grid for grid-stride memory-bound kernels: a multiple of the SM count.
int sm_count();
inline int stream_grid(int64_t work_items, int threads, int ctas_per_sm = 8) {
  int64_t want = ceil_div64(work_items, threads);
  int64_t cap = (int64_t)sm_count() * ctas_per_sm;
  if (want < 1) want = 1;
  return (int)(want < cap ? want : cap);
}


#ifdef __CUDACC__
// ATen's source index for linear modes with align_corners=True
// (area_pixel_compute_scale + compute_source_index_and_lambda): scale = (in-1)/(out-1) in fp32.
struct LinIdx {
  int i0, i1;
  float w0, w1;
};
__device__ __forceinline__ LinIdx lin_index_ac(int dst, float scale, int in_size) {
  LinIdx r;
  const float real = scale * (float)dst;
  int i0 = (int)real;
  if (i0 > in_size - 1) i0 = in_size - 1;
  r.i0 = i0;
  r.i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
  float l1 = real - (float)i0;
  l1 = fminf(fmaxf(l1, 0.0f), 1.0f);
  r.w1 = l1;
  r.w0 = 1.0f - l1;
  return r;
}
// Trilinear pieces in ATen's nesting order with explicit roundings, shared by K4 and the conv kernel that
// up-samples its first source on the fly, so that both produce bit-identical values.
__device__ __forceinline__ float bilerp_hw(float a, float b, float c, float d, float w0, float w1, float h0, float h1) {
  return __fmaf_rn(h1, __fmaf_rn(w1, d, __fmul_rn(w0, c)), __fmul_rn(h0, __fmaf_rn(w1, b, __fmul_rn(w0, a))));
}
__device__ __forceinline__ float lerp_d(float p0, float p1, float d0, float d1) {
  return __fmaf_rn(d1, p1, __fmul_rn(d0, p0));
}
__host__ __device__ __forceinline__ float ac_scale(int in_size, int out_size) {
  return out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.0f;
}
#endif

}  // namespace dram
