/*
 * dram_b200.h — C-ABI of libdram_b200.so: the B200 (sm_100a) device side of the
 * Med3D + dRAM inference hot path of DIAGNijmegen/bodyct-dram-emph-subtype.
 *
 * The reference has no native code: every entry below replaces a call site in
 * the reference's Python that reaches a stock ATen/cuDNN kernel.  The citation
 * on each function names that call site (file:line relative to the reference
 * checkout).
 *
 * Conventions
 *   - every pointer is a raw DEVICE pointer owned by the caller unless the
 *     name says host; nothing here allocates device memory, synchronises the
 *     device or changes the current device (one exception: the
 *     dram_peer_alloc/open/close/free quartet owns the CUDA-IPC exchange
 *     buffers of the SyncBatchNorm kernel);
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous;
 *   - activations are NDHWC bf16 ("channels-last 3-D"), dense maps and
 *     scores are fp32 NCDHW exactly as the reference returns them;
 *   - return value: 0 = DRAM_OK, negative = DRAM_E_*; a message for the last
 *     failure on the calling thread is available from dram_last_error();
 *   - re-entrant; the only global state is per-thread (the error string and
 *     the optional saturation counter) plus the lazily resolved driver entry
 *     point for tensor-map encoding.
 */
#ifndef DRAM_B200_H_
#define DRAM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRAM_OK 0
#define DRAM_E_ARG (-1)     /* bad argument / unsupported shape            */
#define DRAM_E_ARCH (-2)    /* device is not sm_100                         */
#define DRAM_E_LAUNCH (-3)  /* CUDA launch / runtime error                  */
#define DRAM_E_DRIVER (-4)  /* cuTensorMapEncodeTiled unavailable / failed  */

#define DRAM_ABI_VERSION 5

/* 16-bit storage type of activations and packed weights (same layout, same tensor-core rate). */
#define DRAM_DTYPE_BF16 0
#define DRAM_DTYPE_F16 1

/* K1 has two kernels behind one entry point:
 *   TILES  - one TMA box per (filter tap, 64-channel chunk): any filter/stride/dilation, any Cout;
 *   PLANES - 3x3x3 / stride 1 / dilation 1 / pad 1 with Cout 32 or 64: input planes stream once
 *            through a shared-memory ring and the 27 taps read them as shifted UMMA views, each
 *            weight tile feeding four accumulators (operand traffic /7 for the decoder layers). */
#define DRAM_CONV_ALGO_AUTO 0
#define DRAM_CONV_ALGO_TILES 1
#define DRAM_CONV_ALGO_PLANES 2
#define DRAM_CONV_EPILOGUE_AUTO 0
#define DRAM_CONV_EPILOGUE_DIRECT 1
#define DRAM_CONV_EPILOGUE_STAGED 2

/* ---- library ---------------------------------------------------------- */
int dram_version(void);
/* Copies the calling thread's last error text (NUL terminated) into buf. */
int dram_last_error(char *buf, size_t len);
/* Number of SMs of the current device (persistent-grid sizing). */
int dram_sm_count(void);
/* fp16 range probe.  With DRAM_DTYPE_F16 storage the convolution epilogues convert with a saturating
 * cvt (values beyond +-65504 are clamped, never inf).  While a device counter (one uint32, zeroed by the
 * caller) is registered for the calling thread, every convolution launched from that thread (dram_conv3d_run,
 * dram_stem_conv7) adds the number of 32-channel output groups that were clamped (or NaN).  NULL (the default)
 * switches the probe off; the pointer is thread-local state like the error string and is read at launch time,
 * so a CUDA-graph capture taken while it is NULL contains no probe.  Replaces nothing in the reference: its
 * fp32 activations (med3d.py:369-388) cannot overflow; this is the guard for the 16-bit storage choice. */
int dram_set_saturation_counter(void *counter_u32);

/* ---- K1: conv3d implicit GEMM on tcgen05/TMEM, fed by TMA -------------- */
/*
 * Replaces every nn.Conv3d + BatchNorm3d(eval) + ReLU (+ residual add,
 * + shortcut-A) of the network:
 *   med3d.py:93-100 (conv3x3x3), 152-157 (Bottleneck convs), 129-144 and
 *   164-184 (block forward: bn, relu, `out += residual`), 103-112 (shortcut
 *   A), 67/76 (decoder convs, bias=True), 85-89 (crop_concat as a second
 *   K-source), 226-233 / 325-332 (us3 + fcs heads), 382 (sigmoid).
 * The stem (med3d.py:296-304) runs through the same kernel after
 * dram_stem_expand() has unfolded (kh,kw) into 64 pseudo-channels.
 *
 * GEMM view: M = N*Do*Ho*Wo output voxels (tiles of tw*th*td = 128 voxels),
 * N = Cout, K = taps * (C1 + C2).  Weights are packed by the caller as bf16
 * [Cout][kd][kh][kw][C1+C2] (K-major) with the eval BatchNorm scale folded in;
 * `bias` is the folded fp32 per-channel shift.
 */
typedef struct dram_conv_desc {
  /* input geometry (source 1; source 2, if any, has identical N,D,H,W) */
  int32_t n, di, hi, wi;
  int32_t c1;          /* channels of source 1, multiple of 64               */
  int32_t c2;          /* channels of source 2 (concat after source 1), or 0 */
  /* filter */
  int32_t cout;        /* multiple of 32                                     */
  int32_t kd, kh, kw;  /* filter extent per axis (1, 3 or 7)                 */
  int32_t sd, sh, sw;  /* stride                                             */
  int32_t dd, dh, dw;  /* dilation                                           */
  int32_t pd, ph, pw;  /* zero padding                                       */
  /* epilogue */
  int32_t relu;        /* 1: clamp at zero after bias (+ residual)           */
  int32_t res_c;       /* residual channels (<= cout), 0 = none.  Channels   */
                       /* >= res_c get no residual: shortcut type A          */
  int32_t res_stride;  /* residual is read at (d,h,w)*res_stride             */
  int32_t res_d, res_h, res_w; /* residual tensor spatial dims               */
  /* fused 1x1x1 heads (only with cout == 32): out_k = act(W_k . y + b_k)    */
  int32_t n_heads;     /* 0 = none; else 1..2 head groups                    */
  int32_t head_ch[2];  /* channels per head group (1 for reg; 6,3 for cls)   */
  int32_t head_sigmoid;/* 1: sigmoid (med3d.py:382); 0: raw logits (:283)    */
  int32_t store_out;   /* 0: do not write the bf16 activation (heads only)   */
  /* tile shape chosen by the caller (tw*th*td must be 128); 0 = library     */
  /* picks the shape with the fewest tiles                                   */
  int32_t tw, th, td;
  int32_t dtype;       /* DRAM_DTYPE_BF16 or DRAM_DTYPE_F16: type of src/weight/residual/out */
  int32_t algo;        /* DRAM_CONV_ALGO_*: AUTO picks PLANES when the shape allows it         */
  int32_t src1_up2x;   /* 1: src1 is [n][di/2][hi/2][wi/2][c1] and is up-sampled x2 (trilinear,    */
                       /* align_corners=True; med3d.py:83,86) inside the kernel; di,hi,wi stay the  */
                       /* full-resolution dims.  PLANES kernel, cout == 64, c2 > 0 only             */
  int32_t epilogue;    /* TILES kernel: DRAM_CONV_EPILOGUE_AUTO (0: staged for 1x1x1 filters), _DIRECT (1: one */
                       /* 16-byte store per lane and row, BLOCK_N up to 256) or _STAGED (2: 128 x 64 tiles     */
                       /* through shared memory + TMA stores, BLOCK_N <= 128; 1x1x1 filters only)              */
} dram_conv_desc;

typedef struct dram_conv_plan dram_conv_plan; /* opaque: tensor maps + launch geometry */

/* Output spatial size of the convolution described by d. */
int dram_conv3d_out_dims(const dram_conv_desc *d, int32_t *dout, int32_t *hout, int32_t *wout);

/*
 * Builds the TMA tensor maps for the given device buffers and freezes the
 * launch geometry.  Buffers must stay valid and fixed until plan_destroy.
 *   src1, src2 : 16-bit NDHWC inputs (src2 may be NULL when c2 == 0)
 *   weight     : bf16 [cout][taps*(c1+c2)]
 *   bias       : fp32 [cout]
 *   scale      : optional fp32 [cout]; y = acc * scale + bias (lets the caller keep packed weights
 *                in the normal range of the 16-bit type); NULL = 1
 *   residual   : 16-bit NDHWC [n][res_d][res_h][res_w][res_c] or NULL
 *   out        : 16-bit NDHWC [n][do][ho][wo][cout] (may be NULL if !store_out)
 *   head_w     : fp32 [sum(head_ch)][32], head_b fp32 [sum(head_ch)]
 *   head_out   : fp32 NCDHW [n][head_ch[k]][do][ho][wo] per head group
 */
int dram_conv3d_plan_create(const dram_conv_desc *d, const void *src1, const void *src2,
                            const void *weight, const float *bias, const float *scale,
                            const void *residual, void *out, const float *head_w,
                            const float *head_b, float *head_out0, float *head_out1,
                            dram_conv_plan **plan);
int dram_conv3d_plan_destroy(dram_conv_plan *plan);
/* Launches the persistent kernel (grid = min(tiles, max_ctas or #SMs)). */
int dram_conv3d_run(const dram_conv_plan *plan, int32_t max_ctas, void *stream);
/* Introspection for tests / roofline accounting. */
int dram_conv3d_plan_info(const dram_conv_plan *plan, int64_t *flops, int32_t *m_tiles,
                          int32_t *n_tiles, int32_t *block_n, int32_t *stages);
/* FLOPs the plan's kernel really issues to the tensor pipe per run: 2 * 128 * BLOCK_N * 64 for every (tile, tap,
 * 64-channel chunk) stage it executes.  Differs from the algorithmic 2*M*N*K of dram_conv3d_plan_info by the taps
 * skipped inside the zero padding (dilated layers: fewer) and by the padding of border tiles (more). */
int dram_conv3d_plan_executed_flops(const dram_conv_plan *plan, int64_t *flops);
/* Work unit of the tile kernels: a brick of bw x bh x bd output voxels of bn samples (bn > 1: the batch is folded
 * into the brick), run as one 128-row MMA operand or, pair != 0, as two (the M256 kernel).  m_tiles of
 * dram_conv3d_plan_info counts these bricks.  Plane-ring plans report zeros. */
int dram_conv3d_plan_brick(const dram_conv_plan *plan, int32_t *bw, int32_t *bh, int32_t *bd, int32_t *bn,
                           int32_t *pair);
/* Tile order.  When a plan's bricks execute different numbers of taps (padding skipped at the borders of a dilated
 * filter), its persistent kernels balance better walking the tiles by descending cost.  order_size gives the int32
 * entries of that permutation (0: the tiles all cost the same, no order).  set_order builds it on `stream` into the
 * caller's device buffer `order` (one small kernel; no allocation, no synchronisation, graph-capturable) and makes the
 * plan's runs walk it; the buffer must stay alive and unchanged until plan_destroy.  Without it the tiles run in index
 * order, with the same results. */
int dram_conv3d_plan_order_size(const dram_conv_plan *plan, int32_t *entries);
int dram_conv3d_plan_set_order(dram_conv_plan *plan, int32_t *order, void *stream);
/*
 * Work lists (decoder_mask.cu): a run restricted to the work items whose output box, grown by `radius` voxels, meets
 * the support bit mask of dram_decoder_support, whose grid must be the plan's output grid.  Only the 64-channel
 * plane-ring kernel with its sources at full resolution and the 64 -> 32 streaming kernel take a list:
 * dram_conv3d_worklist_size gives 0 for every other plan, otherwise the number of work items (the capacity of
 * `items`; `flags` is scratch of as many bytes).  dram_conv3d_worklist writes the ascending item indices and their
 * number to device memory; dram_conv3d_run_listed reads both on the device (the grid is that of dram_conv3d_run, so
 * the launch is graph-capturable) and computes every listed item exactly as dram_conv3d_run does.
 */
int dram_conv3d_worklist_size(const dram_conv_plan *plan, int32_t *entries);
int dram_conv3d_worklist(const dram_conv_plan *plan, const uint32_t *support, int32_t radius, uint8_t *flags,
                         int32_t *items, int32_t *count, void *stream);
int dram_conv3d_run_listed(const dram_conv_plan *plan, const int32_t *items, const int32_t *count, int32_t max_ctas,
                           void *stream);


/* ---- K2a: stem unfold (feeds K1 with taps 7x1x1, stride 2x1x1) --------- */
/*
 * med3d.py:296-304,371 conv1 = Conv3d(1,64,k7,s2,p3).  Writes
 *   out[n][d][h'][w'][kh*8+j] = x[n][d][2h'-3+kh][2w'-3+j]   (0 outside, 0 for kh==7 or j==7)
 * as bf16, so that the 7^3 stride-2 convolution becomes a 7x1x1 convolution
 * over 64 pseudo-channels.  x is fp32 [n][d][h][w] (the predict_step
 * `image`, models.py:432), h' = (h-1)/2+1, w' = (w-1)/2+1.
 */
int dram_stem_expand(const float *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                     int32_t dtype, void *stream);

/* ---- K2: fused stem, conv1 + bn1 + relu straight from the fp32 image ---- */
/*
 * med3d.py:296-304, 371-373: Conv3d(1, 64, k7, s2, p3, bias=False) + BatchNorm3d(eval) + ReLU.
 * One tcgen05 kernel: producer warps unfold kw of each input plane into shared memory once, kh/kd
 * are shifted UMMA views / accumulation steps, the 7x64x64 weights stay resident (no unfolded copy
 * of the volume in HBM, unlike dram_stem_expand + dram_conv3d_run).
 *   x      : fp32 [n][d][h][w] (the predict_step `image`, models.py:432)
 *   weight : 16-bit, dram_stem_weight_bytes() bytes: even kd [kh=8][kd=6,4,2,0][cout=64][j=8] followed by
 *            odd kd [kh=8][kd=5,3,1][cout=64][j=8]; element = w[cout][0][kd][kh][j-1] * bn_scale for kh < 7
 *            and j >= 1, else 0 (ops.pack_stem_weight_fused)
 *   bias   : fp32 [64] folded BN shift; scale: optional fp32 [64] accumulator multiplier
 *   out    : 16-bit NDHWC [n][(d-1)/2+1][(h-1)/2+1][(w-1)/2+1][64]
 */
size_t dram_stem_weight_bytes(void);
int dram_stem_conv7(const float *x, const void *weight, const float *bias, const float *scale,
                    void *out, int32_t n, int32_t d, int32_t h, int32_t w, int32_t relu,
                    int32_t dtype, int32_t max_ctas, void *stream);
/*
 * The same kernel fed straight from the int16 HU volume: IntensityWindow + Standardize
 * (functional.py:13-26, intensity_transforms.py:104-114; wired at models.py:60-61) collapse to a table —
 * the window clamps every voxel to one of hi - lo + 1 integer values (851 for [-1150, -300]) — that
 * dram_window_lut fills per volume with K8's own arithmetic; the producers clamp and gather.  The values
 * are exactly those of dram_window_standardize; the standardised fp32 image is never written to or re-read
 * from HBM.
 *   hu  : int16 [n][d][h][w];  lut: fp32 [n][lut_size], entry i = standardised value of HU lut_lo + i
 */
#define DRAM_WINDOW_LUT_MAX 4096
int dram_stem_conv7_hu(const int16_t *hu, const float *lut, int32_t lut_lo, int32_t lut_size,
                       const void *weight, const float *bias, const float *scale, void *out, int32_t n,
                       int32_t d, int32_t h, int32_t w, int32_t relu, int32_t dtype, int32_t max_ctas,
                       void *stream);


/* ---- K3: max-pool 3x3x3 stride 2 pad 1 (med3d.py:305, 374) ------------- */
int dram_maxpool3d(const void *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                   int32_t c, int32_t dtype, void *stream);

/* ---- K4: trilinear x2 up-sampling, align_corners=True (med3d.py:83,86) - */
int dram_upsample2x(const void *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                    int32_t c, int32_t dtype, void *stream);

/*
 * The same operation on the tensor cores (upsample_umma.cu): per 8x4x4 output brick a generated 128 x 96
 * interpolation matrix (fp16) times the 96-voxel source patch, one TMA box in and one TMA store out per
 * 64-channel chunk.  Needs c % 64 == 0; rounds the eight interpolation weights to the storage type (one more
 * half-ulp-scale error on top of the storage rounding of the result).  x and out are fixed in the plan (tensor maps).
 */
typedef struct dram_upsample_plan dram_upsample_plan;
int dram_upsample2x_plan_create(const void *x, void *out, int32_t n, int32_t d, int32_t h, int32_t w,
                                int32_t c, int32_t dtype, dram_upsample_plan **plan);
int dram_upsample2x_plan_destroy(dram_upsample_plan *plan);
int dram_upsample2x_plan_run(const dram_upsample_plan *plan, int32_t max_ctas, void *stream);
/* Work lists of the 8x4x4 output bricks, as dram_conv3d_worklist* (the support grid is the output grid). */
int dram_upsample2x_worklist_size(const dram_upsample_plan *plan, int32_t *entries);
int dram_upsample2x_worklist(const dram_upsample_plan *plan, const uint32_t *support, int32_t radius, uint8_t *flags,
                             int32_t *tiles, int32_t *count, void *stream);
int dram_upsample2x_plan_run_listed(const dram_upsample_plan *plan, const int32_t *tiles, const int32_t *count,
                                    int32_t max_ctas, void *stream);

/* ---- support of the dRAM on the decoder grid (decoder_mask.cu) ---------- */
/*
 * K7 reads the dense maps [n][d][h][w] only at the trilinear (align_corners=True) corners {i0, i1} per axis of the
 * ess voxels (i1 included where its weight is 0).  Writes that set as bits: support[((s*d + z)*h + y)*words + x/32]
 * bit x%32, words = ceil(w/32).  ess: uint8 [n][D][H][W]; rows: scratch of n*D*H*words uint32.
 */
int dram_decoder_support(const uint8_t *ess, int32_t n, int32_t D, int32_t H, int32_t W, int32_t d, int32_t h,
                         int32_t w, uint32_t *rows, uint32_t *support, void *stream);

/* ---- K13: the commuted convolution of an up-sampled tensor (med3d.py:83-89, first conv of us1) ---- */
/*
 * UpsampleConvBlock5d.forward up-samples x4 (512 / 2048 channels) x2, concatenates the skip tensor and runs a
 * 3x3x3 convolution with 64 outputs.  Up-sampling acts on space, the filter's channel mixing on channels, so
 *   conv(up(x), W)[o] = sum_tap up(z_tap)[o + tap],   z_tap = W_tap . x  (27 1x1x1 products at LOW resolution,
 *   one dram_conv3d_run with 27*64 output channels, tap-major),
 * and the gather separates per axis.  dram_upconv_axis does one axis:
 *   in  : 16-bit [outer][l_lo][inner][in_channels], the first groups*3*64 channels of a position being
 *         [groups][3 taps of this axis][64]
 *   out : 16-bit [outer][l_hi][inner][groups][64],  l_hi = 2*l_lo in the network (any l_hi works)
 *   out[.., o, .., g, c] = sum_{t<3, 0 <= o+t-1 < l_hi} lerp(in[.., ., .., g, t, c])(o + t - 1)   (align_corners=True
 *   source index and weights of ATen; positions outside the volume are the convolution's zero padding).
 * W pass: outer = N*Dl*Hl, inner = 1, groups = 9; H pass: outer = N*Dl, inner = W, groups = 3; D pass: outer = N,
 * inner = H*W, groups = 1 -> the 64-channel NDHWC tensor that enters the skip half's convolution as its residual.
 */
int dram_upconv_axis(const void *in, void *out, int64_t outer, int32_t l_lo, int32_t l_hi, int64_t inner,
                     int32_t groups, int32_t in_channels, int32_t dtype, void *stream);

/* ---- K6: lobe-masked / global pooling (med3d.py:383-387, 284) ---------- */
/*
 * dense: fp32 [n][ch][d][h][w].  mask: [n][md][mh][mw], uint8 (non-zero = lung)
 * or, with mask_is_f32 != 0, fp32 weights exactly as `dout * lungs` uses them,
 * resampled on the fly with ATen's legacy `nearest` rule (med3d.py:386), or
 * NULL for the unmasked mean (lungs=None, med3d.py:383-384 and the cls path).
 * out: fp32 [n][ch]  = sum(dense*mask)/sum(mask)  (or the plain mean).
 * workspace: at least dram_pool_workspace_bytes(n, ch) bytes.
 */
size_t dram_pool_workspace_bytes(int32_t n, int32_t ch);
int dram_masked_pool(const float *dense, const void *mask, int32_t mask_is_f32, float *out,
                     void *workspace, int32_t n, int32_t ch, int32_t d, int32_t h, int32_t w,
                     int32_t md, int32_t mh, int32_t mw, void *stream);

/* ---- K7: dRAM = trilinear(dense -> scan size, align_corners) * ess ----- */
/*
 * models.py:438-441 (predict_step).  dense0/dense1: fp32 [n][1][d][h][w];
 * ess, lungs: uint8 [n][D][H][W]; out0/out1: fp32 [n][1][D][H][W];
 * pct: fp32 [2][n] = sum_b(out_k[b]) / sum over the WHOLE batch of lungs
 * (reference quirk Q1) or per sample when per_sample_denominator != 0.
 */
size_t dram_dram_workspace_bytes(int32_t n);
int dram_dram_upsample_mask(const float *dense0, const float *dense1, const uint8_t *ess,
                            const uint8_t *lungs, float *out0, float *out1, float *pct,
                            void *workspace, int32_t n, int32_t d, int32_t h, int32_t w,
                            int32_t D, int32_t H, int32_t W, int32_t per_sample_denominator,
                            void *stream);

/* ---- K7l: lesion percentages per label (per lobe) of both dRAM maps ----- */
/*
 * Not in the reference (it reports whole-lung numbers only).  map0/map1: fp32 [n][count] (the K7 outputs
 * [n][1][D][H][W]); ess, labels: uint8 [n][count] (labels: lobe labels resized like the masks).
 *   voxels[b][k]  int64 [n][256] = #{v : labels[b][v] == k}                                (exact)
 *   pct[m][b][k]  fp32 [2][n][256] = (float)S / (float)voxels[b][k],
 *                 S = sum over {v : labels[b][v] == k and ess[b][v] != 0} of map_m[b][v] in fp64
 *                 (the conversion of K7's percentages; NaN where voxels[b][k] == 0)
 * The denominator is always the sample's own label volume.  Bit-reproducible: per-CTA partials and a
 * fixed-order finish, no floating-point atomics.  Map values are read only where ess is set.  ess and
 * labels that start on a 16-byte boundary with count % 16 == 0 take 16-byte loads, anything else a byte
 * path.  workspace: dram_lobe_workspace_bytes(n, count) bytes, 8-byte aligned; count < 2^31.
 */
size_t dram_lobe_workspace_bytes(int32_t n, int64_t count);
int dram_lobe_sums(const float *map0, const float *map1, const uint8_t *ess, const uint8_t *labels, float *pct,
                   int64_t *voxels, void *workspace, int32_t n, int64_t count, void *stream);

/* ---- K8: HU window + standardise (functional.py:13-26,                   */
/*          intensity_transforms.py:104-114; wired at models.py:60-61) ---- */
/*
 * hu: int16 [count]; out: fp32 [count] = (v - mean(v)) / std_unbiased(v) with
 * v = (clamp(hu, lo, hi) - lo) / (hi - lo) in fp32.  One volume per call
 * (statistics are per volume).  stats_out (optional, fp32[2]) = mean, std.
 * Buffers of any alignment are accepted (16-byte aligned ones take the vector path).
 */
size_t dram_preprocess_workspace_bytes(void);
int dram_window_standardize(const int16_t *hu, float *out, float *stats_out, void *workspace,
                            int64_t count, float lo, float hi, void *stream);
/*
 * Batched forms: n volumes of `count` voxels each, stored back to back ([n][count]); statistics stay per
 * volume.  Three launches whatever n is (statistics of all volumes, finalize, apply).  stats_out: fp32 [n][2].
 * dram_window_stats runs the statistics pass only; dram_window_lut adds the per-volume table
 * lut[v][i] = standardised value of HU (int)lo + i, i in [0, hi - lo] (integral lo/hi, at most
 * DRAM_WINDOW_LUT_MAX entries) that dram_stem_conv7_hu gathers from.  Workspace:
 * dram_preprocess_workspace_bytes_n(n) bytes, 8-byte aligned.  Volumes that do not start on a 16-byte
 * boundary (count % 8 != 0, or an unaligned base) take a scalar path instead of failing.
 */
size_t dram_preprocess_workspace_bytes_n(int32_t n);
int dram_window_standardize_batch(const int16_t *hu, float *out, float *stats_out, void *workspace,
                                  int32_t n, int64_t count, float lo, float hi, void *stream);
int dram_window_stats(const int16_t *hu, float *stats_out, void *workspace, int32_t n, int64_t count,
                      float lo, float hi, void *stream);
int dram_window_lut(const int16_t *hu, float *lut, float *stats_out, void *workspace, int32_t n,
                    int64_t count, float lo, float hi, void *stream);

/* ---- K8b: Interpolate transform (spatial_transforms.py:55-97) ---------- */
/*
 * Image: in-plane bilinear (align_corners=True) to (H2,W2) then slice pick
 * d_idx[k] (the caller builds d_idx with torch.linspace(0,D-1,D2).long(),
 * spatial_transforms.py:66).  Mask: in-plane legacy nearest + same slice pick.
 * Labels: the voxel the mask rule picks, its value kept instead of cast to 0/1 (lobe labels; not in
 * the reference), so (labels_out > 0) equals the mask resize of (labels > 0) bit for bit.
 */
int dram_resize_image(const float *x, float *out, const int32_t *d_idx, int32_t D, int32_t H,
                      int32_t W, int32_t D2, int32_t H2, int32_t W2, void *stream);
int dram_resize_mask(const uint8_t *x, uint8_t *out, const int32_t *d_idx, int32_t D, int32_t H,
                     int32_t W, int32_t D2, int32_t H2, int32_t W2, void *stream);
int dram_resize_labels(const uint8_t *x, uint8_t *out, const int32_t *d_idx, int32_t D, int32_t H,
                       int32_t W, int32_t D2, int32_t H2, int32_t W2, void *stream);

/* ---- f1: device pre-steps of SubtypingInference.get_data (dataset.py:66-80) ---- */
/*
 * dram_mask_bbox: bbox (device int32[6]) = {zmin, zmax+1, ymin, ymax+1, xmin, xmax+1} of mask != 0
 * ({D,0,H,0,W,0} for an empty mask) — scipy.ndimage.find_objects(mask > 0)[0] of utils.py:54.  The
 * caller grows it by ceil(border / spacing) and clips (utils.py:55-60).
 */
int dram_mask_bbox(const uint8_t *mask, int32_t D, int32_t H, int32_t W, int32_t *bbox, void *stream);
/*
 * dram_lung_crop: for the crop window [z0,z0+cd) x [y0,y0+ch) x [x0,x0+cw) of a D x H x W scan
 *   lung    = lobe > 0                                                   (dataset.py:67)
 *   dlung   = binary_dilation(lung, 3x3x3 full structure, iterations=2)  (:68; a 5x5x5 box maximum
 *             over the WHOLE volume with a zero border, not just the crop)
 *   image_c = dlung ? scan : -2048                                        (:69, :71)
 *   lung_c  = lung                                                        (:72, :77)
 *   ess_c   = (image_c < -910) & lung                                     (:78)
 * scan int16, lobe uint8 (labels), outputs int16 / uint8 / uint8 of the crop size; workspace of
 * dram_lung_crop_workspace_bytes(cd, ch, cw) bytes.  Bit-exact.
 */
size_t dram_lung_crop_workspace_bytes(int32_t cd, int32_t ch, int32_t cw);
int dram_lung_crop(const int16_t *scan, const uint8_t *lobe, int32_t D, int32_t H, int32_t W, int32_t z0,
                   int32_t y0, int32_t x0, int32_t cd, int32_t ch, int32_t cw, int16_t *image_c,
                   uint8_t *lung_c, uint8_t *ess_c, void *workspace, void *stream);
/*
 * Densitometry on the full-resolution grid (not in the reference): the same device scan and uint8 lobe
 * labels the two calls above read, count voxels.  Both calls zero their own outputs, keep privatised
 * per-CTA counters in shared memory and add them into the int64 outputs with integer atomics, so the
 * result is exact and the same in any order.  Labels that start on a 16-byte boundary take 16-byte loads
 * (the scan too, for the histograms); other views and the last count % 16 voxels take a byte path.
 * 0 <= count < 2^31.  No host synchronisation and no host-to-device copy: both are graph-capturable.
 *
 * dram_label_counts: counts (device int64 [256])[k] = #{v : labels[v] == k}.
 */
int dram_label_counts(const uint8_t *labels, int64_t count, int64_t *counts, void *stream);
/*
 * dram_label_hu_hist: HU histograms of up to 16 labels in one pass.  slot_of_label is a HOST array of
 * 256 bytes (passed to the kernel by value): the slot 0 .. nslots-1 label k goes to, or 0xFF for a label
 * that is not tracked.  1 <= nslots <= 16.  For every slot s (outputs device int64):
 *   hist[s][b]  = #{v : slot_of_label[labels[v]] == s and clamp(scan[v], -1024, 1023) == b - 1024}
 *   hu_sum[s]   = sum of scan[v] (unclamped) over the same voxels
 * The scan is read only for 16-voxel vectors that hold a tracked label.
 */
int dram_label_hu_hist(const int16_t *scan, const uint8_t *labels, int64_t count, const uint8_t *slot_of_label,
                       int32_t nslots, int64_t *hist, int64_t *hu_sum, void *stream);

/* ---- f2: device post-processing of one scan (processor.py:111-158, utils.py:28-37) ---- */
/*
 * out uint8 [OD][OH][OW] = 0 outside the crop window; inside,
 *   trunc(clip(trilinear_align_corners(map [d][h][w] -> [cd][ch][cw]), 0, 1) * 255.0)   (fp64 product)
 * i.e. F.interpolate(size=recon_size) -> paste into np.zeros(original_size) -> windowing((0,1)) ->
 * astype(uint8), in one pass; only uint8 has to leave the GPU.
 */
int dram_heatmap_u8(const float *map, int32_t d, int32_t h, int32_t w, uint8_t *out, int32_t OD, int32_t OH,
                    int32_t OW, int32_t z0, int32_t y0, int32_t x0, int32_t cd, int32_t ch, int32_t cw,
                    void *stream);

/* ---- K9: conv3d weight gradient (training path, SURVEY 8f f4) ------------ */
/*
 * The reference has no backward code of its own: train.py (Lightning automatic optimisation,
 * models.py:495-582) differentiates every nn.Conv3d of med3d.py:93-100, 67/76, 152-157 through
 * autograd.  This entry computes what autograd leaves in `conv.weight.grad`:
 *   dw[cout][cin_offset + ci][kd][kh][kw] (+)= sum_v dy[v][cout] * x[v*stride + tap*dilation - pad][ci]
 * on the tensor cores (both operands MN-major straight from NDHWC, fp32 accumulation in TMEM, K split
 * over the voxels with a deterministic second pass).  Only the geometry fields of the descriptor are read:
 * n, di, hi, wi, c1 (channels of x, multiple of 64; c2 must be 0), cout (32, 64, 128, 256 or a multiple
 * of 256), k*, s*, d*, p*, dtype.
 *   x  : 16-bit NDHWC [n][di][hi][wi][c1]   (the convolution's input, or one source of a concatenation)
 *   dy : 16-bit NDHWC [n][do][ho][wo][cout] (gradient of the convolution's output)
 *   dw : fp32 [cout][cin_total][kd][kh][kw] (PyTorch's weight layout); this call fills the channel range
 *        [cin_offset, cin_offset + c1) — a concatenated input (med3d.py:87) is two calls
 *   workspace : dram_conv3d_wgrad_workspace_bytes(d) bytes (negative return: bad descriptor)
 * run(): accumulate != 0 adds to dw instead of overwriting it.
 */
typedef struct dram_wgrad_plan dram_wgrad_plan;
int64_t dram_conv3d_wgrad_workspace_bytes(const dram_conv_desc *d);
int dram_conv3d_wgrad_plan_create(const dram_conv_desc *d, const void *x, const void *dy, float *dw,
                                  int32_t cin_total, int32_t cin_offset, void *workspace,
                                  int64_t workspace_bytes, dram_wgrad_plan **plan);
int dram_conv3d_wgrad_plan_destroy(dram_wgrad_plan *plan);
int dram_conv3d_wgrad_plan_info(const dram_wgrad_plan *plan, int64_t *flops, int32_t *items, int32_t *kslices,
                                int32_t *block_n);
int dram_conv3d_wgrad_run(const dram_wgrad_plan *plan, int32_t accumulate, int32_t max_ctas, void *stream);

/* ---- K10: train-mode BatchNorm3d (+ReLU, +residual), forward and backward (SURVEY 8f f4) ---- */
/*
 * What autograd sees of bn(conv(x)) / relu / `out += residual` (med3d.py:129-144, 164-184, 74-80, 371-373) when the
 * reference trains (model.train(), train.py).  x, res, y, dy, dx, dres: 16-bit NDHWC viewed as [m][c] rows,
 * c a multiple of 8 with 256 % (c/8) == 0 (8 ... 2048).  All per-channel vectors fp32 [c]; sums fp64 [2][c].
 *   dram_bn_stats            sums = {sum x, sum x^2} over the m rows (two-phase, deterministic)
 *   -- the caller may all-reduce `sums` over the process group here (SyncBatchNorm, train.py:101) --
 *   dram_bn_finalize         mean, rstd = 1/sqrt(var_biased + eps); scale = gamma*rstd; shift = beta - mean*scale;
 *                            running_mean/var (may be NULL) updated with `momentum`, unbiased variance
 *   dram_bn_apply            out = act(x*scale + shift (+ res)),  act = ReLU if relu != 0
 *   dram_bn_backward_reduce  sums = {sum dz, sum dz*xhat}, dz = dy where y > 0 (y = forward output; NULL: no ReLU)
 *   dram_bn_backward_apply   dx = gamma*rstd*(dz - sums[0]/count - xhat*sums[1]/count); dres = dz (may be NULL)
 * dgamma = sums[1], dbeta = sums[0] of the backward reduction.  workspace: dram_bn_workspace_bytes(c) bytes.
 */
int64_t dram_bn_workspace_bytes(int32_t c);
int dram_bn_stats(const void *x, int64_t m, int32_t c, int32_t dtype, double *sums, void *workspace, void *stream);
int dram_bn_finalize(const double *sums, double count, const float *gamma, const float *beta, float eps,
                     float momentum, float *running_mean, float *running_var, float *scale, float *shift,
                     float *mean, float *rstd, int32_t c, void *stream);
int dram_bn_apply(const void *x, const float *scale, const float *shift, const void *res, int32_t relu, void *out,
                  int64_t m, int32_t c, int32_t dtype, void *stream);
int dram_bn_backward_reduce(const void *dy, const void *x, const void *y, const float *mean, const float *rstd,
                            int64_t m, int32_t c, int32_t dtype, double *sums, void *workspace, void *stream);
int dram_bn_backward_apply(const void *dy, const void *x, const void *y, const float *mean, const float *rstd,
                           const float *gamma, const double *sums, double count, void *dx, void *dres, int64_t m,
                           int32_t c, int32_t dtype, void *stream);

/* ---- K4T / K3T: backward of the x2 up-sampling and of the max-pool (SURVEY 8f f4) ---- */
/*
 * dram_upsample2x_backward: adjoint of K4 (med3d.py:83,86; same ATen index arithmetic): dy [n][2d][2h][2w][c] ->
 *   dx [n][d][h][w][c].  Gather formulation, fp32 accumulation, deterministic.
 * dram_maxpool3d_backward: backward of K3 (med3d.py:305): x [n][d][h][w][c] (the pool's input), dy over the pooled
 *   grid -> dx; a window's gradient goes to its FIRST maximum in (d,h,w) scan order, as ATen's
 *   max_pool3d_with_indices does (ties are the rule after ReLU): an arg-max pass into `workspace`
 *   (dram_maxpool3d_backward_workspace_bytes: one byte per pooled element), then a gather pass.  c multiple of 8
 *   for both.
 */
int dram_upsample2x_backward(const void *dy, void *dx, int32_t n, int32_t d, int32_t h, int32_t w, int32_t c,
                             int32_t dtype, void *stream);
int64_t dram_maxpool3d_backward_workspace_bytes(int32_t n, int32_t d, int32_t h, int32_t w, int32_t c);
int dram_maxpool3d_backward(const void *x, const void *dy, void *dx, void *workspace, int32_t n, int32_t d,
                            int32_t h, int32_t w, int32_t c, int32_t dtype, void *stream);

/* ---- K5T: the two 1x1x1 regression heads + sigmoid in training (med3d.py:329-332, 382) ---- */
/*
 * x : 16-bit NDHWC rows [m][32] (us3's output); w fp32 [2][32] (fcs.0.weight, fcs.1.weight), b fp32 [2].
 * forward : out_k[m] = sigmoid(w_k . x[m] + b_k), fp32 (= the [B,1,D,H,W] dense maps, flat).
 * backward: from s_k = out_k and g_k = d loss / d out_k: dx 16-bit [m][32], dw fp32 [2][32], db fp32 [2];
 *           two-phase deterministic reduction, workspace of dram_heads_workspace_bytes() bytes.
 */
int64_t dram_heads_workspace_bytes(void);
int dram_heads_sigmoid_forward(const void *x, const float *w, const float *b, float *out0, float *out1, int64_t m,
                               int32_t dtype, void *stream);
int dram_heads_sigmoid_backward(const void *x, const float *w, const float *s0, const float *s1, const float *g0,
                                const float *g1, void *dx, float *dw, float *db, void *workspace, int64_t m,
                                int32_t dtype, void *stream);

/* ---- K10x: SyncBatchNorm's statistics exchange over NVLink peer memory (train.py:101 `sync_batchnorm=True`) ---- */
/*
 * One process per GPU on one node (<= 8 ranks).  Start-up, once per rank:
 *   dram_peer_alloc(dram_peer_exchange_bytes(), &own, handle)   cudaMalloc + zero + CUDA IPC handle (64 bytes)
 *   -- exchange the handles between the ranks (e.g. torch.distributed.all_gather_object) --
 *   dram_peer_open(handle_of_rank_r, &peer_r) for every other rank; then a barrier.
 * Per exchange (the all-reduce between dram_bn_stats / dram_bn_backward_reduce and the following pass):
 *   dram_peer_allreduce_f64(in, out, n, peers, world, rank, seq, status, stream)
 *     in/out : fp64 [n] on this rank (n = 2*c <= 4096; may alias), out = sum over the ranks in rank order — every rank
 *              gets the same bits;
 *     peers  : host array of `world` device pointers, peers[rank] = own buffer;
 *     seq    : 1, 2, 3, ... the same sequence on every rank (one per exchange);
 *     status : device int32, 0 = healthy; set non-zero when a peer did not answer within ~60 s, after which every
 *              call copies in -> out without waiting (check it on the host at a convenient point).
 * One kernel pushes the sums into every peer's buffer, raises release flags, waits for the peers' flags and adds.
 * dram_peer_close / dram_peer_free undo open / alloc.  These are the only entry points that own device memory.
 */
#define DRAM_PEER_HANDLE_BYTES 64
int64_t dram_peer_exchange_bytes(void);
int dram_peer_alloc(int64_t bytes, void **ptr, void *handle64);
int dram_peer_open(const void *handle64, void **ptr);
int dram_peer_close(void *ptr);
int dram_peer_free(void *ptr);
int dram_peer_allreduce_f64(const double *in, double *out, int32_t n, void *const *peers, int32_t world, int32_t rank,
                            uint64_t seq, int32_t *status, void *stream);

/* ---- K11: the training loss and its gradient (SURVEY 8f f4) ---- */
/*
 * What ScanRegLightningModule.shared_step(TRAIN) computes from the two sigmoid maps (models.py:547-565) and what
 * autograd returns for them, fused: the lobe-masked means (med3d.py:383-387), `_interval_regression_loss`
 * (models.py:495-506), BinaryDice between the masked maps and the masked BinaryCrossEntropy of clamp(cle + pse, 0, 1)
 * (models.py:508-518, metrics.py:4-47); total = loss_cle + loss_pse + 2 * mul_loss + seg_loss.
 *   cle_map, pse_map : fp32 [b][d2][h2][w2] (the dense outputs, values in (0, 1))
 *   lungs, ems       : 0/1 bytes [b][d][h][w] at scan resolution; sampled with ATen's legacy `nearest` index
 *   cle_labels, pse_labels : int64 [b] (a scan's `ems` counts only if one of its labels is > 0, models.py:553)
 *   *_bands fp32 [b][2] = (lo, hi) of `_generate_regression_labels` (models.py:477-493); *_weights fp32 [b]
 *   coef : fp32 [DRAM_LOSS_COEF_HEAD + 4*b] written by forward, read by backward:
 *          [TOTAL] [CLE] [PSE] [MUL] [SEG] = the loss and its four terms; 5..15 internal;
 *          then per sample {mean of cle_map in the lungs, mean of pse_map in the lungs, 2 internal}
 *          (= reg_outs of med3d.py:387, what `_ratio_to_label` bins, models.py:543-544)
 *   grad_loss : device pointer to d(objective)/d(loss), or NULL for 1
 *   grad_cle, grad_pse : fp32, same shape as the maps
 * Two-phase fixed-order fp64 reduction: results are deterministic.  b <= 64.
 */
#define DRAM_LOSS_COEF_TOTAL 0
#define DRAM_LOSS_COEF_CLE 1
#define DRAM_LOSS_COEF_PSE 2
#define DRAM_LOSS_COEF_MUL 3
#define DRAM_LOSS_COEF_SEG 4
#define DRAM_LOSS_COEF_HEAD 16
int64_t dram_train_loss_workspace_bytes(int32_t b);
int dram_train_loss_forward(const float *cle_map, const float *pse_map, const uint8_t *lungs, const uint8_t *ems,
                            const int64_t *cle_labels, const int64_t *pse_labels, const float *cle_bands,
                            const float *pse_bands, const float *cle_weights, const float *pse_weights, int32_t b,
                            int32_t d, int32_t h, int32_t w, int32_t d2, int32_t h2, int32_t w2, float beta,
                            float gamma, float *coef, void *workspace, void *stream);
int dram_train_loss_backward(const float *cle_map, const float *pse_map, const uint8_t *lungs, const uint8_t *ems,
                             const int64_t *cle_labels, const int64_t *pse_labels, const float *coef,
                             const float *grad_loss, int32_t b, int32_t d, int32_t h, int32_t w, int32_t d2,
                             int32_t h2, int32_t w2, float *grad_cle, float *grad_pse, void *stream);

/* ---- K12: Adam over flat buffers (models.py:685-698 `torch.optim.Adam(self.parameters(), lr=...)`) ---- */
/*
 * One launch updates every parameter: param, grad, exp_avg, exp_avg_sq are fp32 [n], 16-byte aligned (the flat
 * buffers of the training step).  torch.optim.Adam's update with amsgrad off and no weight decay:
 *   g = grad * grad_scale;  m += (1-beta1)(g - m);  v = beta2 v + (1-beta2) g^2;
 *   param -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps),   step = 1, 2, ...
 */
int dram_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, double lr,
                   double beta1, double beta2, double eps, int32_t step, float grad_scale, void *stream);

/* ---- weight re-packing for the training step ---------------------------- */
/*
 * w: fp32 [cout][cin_total][taps] (PyTorch's Conv3d weight, taps = kd*kh*kw) -> 16-bit packed operand of
 *   transpose == 0: K1's layout   out[co][t][ci]          = w[co][cin0+ci][t],            ci < cin_n
 *   transpose != 0: dgrad layout  out[ci][t][co < cout_pad] = w[co][cin0+ci][taps-1-t], zero for co >= cout
 * (the second is the transposed convolution's filter: spatially flipped, channels swapped; backward.pack_dgrad_weight).
 */
int dram_pack_conv_weight(const float *w, void *out, int32_t cout, int32_t cin_total, int32_t taps, int32_t cin0,
                          int32_t cin_n, int32_t transpose, int32_t cout_pad, int32_t dtype, void *stream);

/* ---- layout helpers ---------------------------------------------------- */
/* fp32 NCDHW -> 16-bit NDHWC and back (test / debugging / hook support). */
int dram_ncdhw_f32_to_ndhwc_16(const float *x, void *out, int32_t n, int32_t c, int32_t d,
                               int32_t h, int32_t w, int32_t dtype, void *stream);
int dram_ndhwc_16_to_ncdhw_f32(const void *x, float *out, int32_t n, int32_t c, int32_t d,
                               int32_t h, int32_t w, int32_t dtype, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DRAM_B200_H_ */
