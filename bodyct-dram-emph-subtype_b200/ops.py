"""Torch-facing wrappers of the C-ABI kernels (one function per kernel family of SURVEY §7.1b).

Each wrapper checks shapes/dtypes, allocates the output with torch's caching allocator, passes
raw device pointers plus the current CUDA stream to libdram_b200.so and returns torch tensors.
The stateless kernel families are registered as `torch.library.custom_op`s in the `dram_b200::`
namespace by `custom_ops.py` (imported at the bottom of this module): `torch.ops.dram_b200.conv3d`,
`.stem_conv7`, `.maxpool3d`, `.upsample2x`, `.masked_pool`, `.dram_upsample_mask`, `.window_standardize`,
`.resize_image`, `.resize_mask`, `.heatmap_u8`, `.lobe_scores`, `.label_counts`, `.hu_histograms`, each with a fake
(shape-only) implementation.  The functions below are what those ops call; the engine calls them (and its frozen `Conv3dPlan`s) directly
and replays the whole sequence as one CUDA graph.

Activations are NDHWC 16-bit tensors of shape [N, D, H, W, C]: torch.bfloat16 or torch.float16
(`ACT_DTYPES`; both run at the same tensor-core rate, fp16 carries 3 more mantissa bits).  There
is no CPU path: every function raises on a non-CUDA tensor.
"""
import ctypes as C
import os

import torch

from . import _capi
from ._capi import ConvDesc, check

ACT_DTYPES = {torch.bfloat16: _capi.DRAM_DTYPE_BF16, torch.float16: _capi.DRAM_DTYPE_F16}


def default_act_dtype():
    """Storage type of activations/weights: env DRAM_B200_DTYPE = fp16 (default) | bf16."""
    name = os.environ.get("DRAM_B200_DTYPE", "fp16").lower()
    if name in ("fp16", "f16", "float16", "half"):
        return torch.float16
    if name in ("bf16", "bfloat16"):
        return torch.bfloat16
    raise ValueError(f"DRAM_B200_DTYPE={name!r}: expected fp16 or bf16")


class ActivationOverflow(RuntimeError):
    """A convolution output left the finite fp16 range and was clamped (see dram_set_saturation_counter)."""


def sat_check_mode():
    """env DRAM_B200_SAT_CHECK = first (default: probe the first forward after every weight change) | always | off."""
    mode = os.environ.get("DRAM_B200_SAT_CHECK", "first").lower()
    if mode not in ("first", "always", "off"):
        raise ValueError(f"DRAM_B200_SAT_CHECK={mode!r}: expected first, always or off")
    return mode


def graphs_enabled():
    """env DRAM_B200_GRAPH = 1 (default: the engine replays its launch sequence as one CUDA graph) | 0 (eager)."""
    return os.environ.get("DRAM_B200_GRAPH", "1").lower() not in ("0", "off", "false", "no")


def _need16(t, name, ndim=None):
    if isinstance(t, torch.Tensor) and t.dtype not in ACT_DTYPES:
        raise TypeError(f"{name}: expected bfloat16 or float16, got {t.dtype}")
    return _need(t, t.dtype, name, ndim)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _need(t, dtype, name, ndim=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (libdram_b200 has no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name}: expected {ndim} dims, got shape {tuple(t.shape)}")
    return t


def sm_count():
    return _capi.load().dram_sm_count()


# --------------------------------------------------------------------------------------------
# K1 conv3d
# --------------------------------------------------------------------------------------------
def _triple(v):
    return (v, v, v) if isinstance(v, int) else tuple(v)


class Conv3dPlan:
    """A frozen conv3d launch: TMA tensor maps for fixed buffers + geometry.

    x1 (and optional x2, concatenated after x1 along channels) are NDHWC bf16; `weight` is the
    packed 16-bit [Cout, taps*(C1+C2)] matrix from `pack_conv_weight`; `bias` fp32 [Cout]; the
    optional fp32 `scale` [Cout] multiplies the accumulator before the bias.
    `residual` is NDHWC bf16 with `res_c <= Cout` channels read at `res_stride` (shortcut A).
    `heads = (head_w [sum_ch, 32] fp32, head_b [sum_ch] fp32, (ch0, ch1), sigmoid)` fuses the
    1x1x1 heads into the epilogue of a 32-channel conv.
    `upsample_x1=True`: x1 is [N, D/2, H/2, W/2, C1] and is up-sampled x2 (trilinear, align_corners=True,
    med3d.py:83-86) inside the kernel; x2 (required) is the full-resolution skip tensor.
    """

    def __init__(self, x1, weight, bias, *, x2=None, scale=None, kernel=3, stride=1, dilation=1,
                 padding=None, relu=True, residual=None, res_stride=1, heads=None, store_out=True,
                 out=None, tile=None, algo="auto", upsample_x1=False, epilogue="auto"):
        lib = _capi.load()
        _need16(x1, "conv3d x1", 5)
        adt = x1.dtype
        n, di, hi, wi, c1 = x1.shape
        if upsample_x1:  # x1 is the half-resolution tensor; the kernel up-samples it x2 on the fly
            di, hi, wi = 2 * di, 2 * hi, 2 * wi
        c2 = 0
        if x2 is not None:
            _need(x2, adt, "conv3d x2", 5)
            if tuple(x2.shape[:4]) != (n, di, hi, wi):
                raise ValueError(f"conv3d: x2 {tuple(x2.shape)} does not match x1 {tuple(x1.shape)}")
            c2 = x2.shape[4]
        k, s, dl = _triple(kernel), _triple(stride), _triple(dilation)
        pad = tuple(dl[i] * (k[i] - 1) // 2 for i in range(3)) if padding is None else _triple(padding)
        _need(weight, adt, "conv3d weight", 2)
        _need(bias, torch.float32, "conv3d bias", 1)
        if scale is not None:
            _need(scale, torch.float32, "conv3d scale", 1)
            if scale.shape[0] != weight.shape[0]:
                raise ValueError("conv3d: scale length != cout")
        cout = weight.shape[0]
        taps = k[0] * k[1] * k[2]
        if weight.shape[1] != taps * (c1 + c2):
            raise ValueError(f"conv3d: packed weight K={weight.shape[1]} != taps*(c1+c2)={taps * (c1 + c2)}")
        if bias.shape[0] != cout:
            raise ValueError("conv3d: bias length != cout")

        d = ConvDesc()
        d.n, d.di, d.hi, d.wi, d.c1, d.c2, d.cout = n, di, hi, wi, c1, c2, cout
        d.kd, d.kh, d.kw = k
        d.sd, d.sh, d.sw = s
        d.dd, d.dh, d.dw = dl
        d.pd, d.ph, d.pw = pad
        d.relu = 1 if relu else 0
        d.dtype = ACT_DTYPES[adt]
        d.algo = _capi.CONV_ALGO[algo]
        d.src1_up2x = 1 if upsample_x1 else 0
        d.epilogue = _capi.CONV_EPILOGUE[epilogue]
        if residual is not None:
            _need(residual, adt, "conv3d residual", 5)
            d.res_c = residual.shape[4]
            d.res_stride = res_stride
            d.res_d, d.res_h, d.res_w = residual.shape[1:4]
            if residual.shape[0] != n:
                raise ValueError("conv3d: residual batch mismatch")
        else:
            d.res_stride = 1
        head_w = head_b = None
        if heads is not None:
            head_w, head_b, head_ch, sigmoid = heads
            _need(head_w, torch.float32, "conv3d head_w", 2)
            _need(head_b, torch.float32, "conv3d head_b", 1)
            d.n_heads = len(head_ch)
            for i, ch in enumerate(head_ch):
                d.head_ch[i] = ch
            d.head_sigmoid = 1 if sigmoid else 0
            if head_w.shape != (sum(head_ch), 32) or head_b.shape[0] != sum(head_ch):
                raise ValueError("conv3d: head weight/bias shape mismatch")
        d.store_out = 1 if store_out else 0
        if tile is not None:
            d.tw, d.th, d.td = tile

        do, ho, wo = C.c_int32(), C.c_int32(), C.c_int32()
        check(lib.dram_conv3d_out_dims(C.byref(d), C.byref(do), C.byref(ho), C.byref(wo)), "dram_conv3d_out_dims")
        self.out_shape = (n, do.value, ho.value, wo.value, cout)
        if store_out:
            if out is None:
                out = torch.empty(self.out_shape, dtype=adt, device=x1.device)
            else:
                _need(out, adt, "conv3d out", 5)
                if tuple(out.shape) != self.out_shape:
                    raise ValueError(f"conv3d: out shape {tuple(out.shape)} != {self.out_shape}")
        else:
            out = None
        self.out = out
        self.head_outs = []
        if heads is not None:
            for ch in heads[2]:
                self.head_outs.append(torch.empty((n, ch, do.value, ho.value, wo.value), dtype=torch.float32,
                                                  device=x1.device))
        ho0 = self.head_outs[0] if len(self.head_outs) > 0 else None
        ho1 = self.head_outs[1] if len(self.head_outs) > 1 else None

        handle = C.c_void_p()
        check(lib.dram_conv3d_plan_create(C.byref(d), _p(x1), _p(x2), _p(weight), _p(bias), _p(scale),
                                          _p(residual), _p(out), _p(head_w), _p(head_b), _p(ho0), _p(ho1),
                                          C.byref(handle)), "dram_conv3d_plan_create")
        self._handle = handle
        self._lib = lib
        # keep every buffer the tensor maps point at alive for the life of the plan
        self._keep = (x1, x2, weight, bias, scale, residual, out, head_w, head_b, ho0, ho1)
        flops, mt, nt, bn, st = C.c_int64(), C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        check(lib.dram_conv3d_plan_info(handle, C.byref(flops), C.byref(mt), C.byref(nt), C.byref(bn),
                                        C.byref(st)), "dram_conv3d_plan_info")
        self.flops, self.m_tiles, self.n_tiles, self.block_n, self.stages = (
            flops.value, mt.value, nt.value, bn.value, abs(st.value))
        self.algo = "planes" if st.value < 0 else "tiles"
        ex = C.c_int64()
        check(lib.dram_conv3d_plan_executed_flops(handle, C.byref(ex)), "dram_conv3d_plan_executed_flops")
        self.executed_flops = ex.value   # tap skipping and tile padding included (what the tensor pipe really does)
        self.desc = d

    def run(self, max_ctas=0):
        check(self._lib.dram_conv3d_run(self._handle, max_ctas, _stream()), "dram_conv3d_run")
        return self.out

    def worklist_size(self):
        """Number of work items if the plan's kernel takes a work list (`run_listed`), else 0."""
        n = C.c_int32()
        check(self._lib.dram_conv3d_worklist_size(self._handle, C.byref(n)), "dram_conv3d_worklist_size")
        return n.value

    def build_worklist(self, support, radius, flags, items, count):
        """Items whose output box grown by `radius` meets `support` (`decoder_support` on the output grid) ->
        items int32 [worklist_size()] (ascending) and count int32 [1], on the device; flags: uint8 scratch."""
        check(self._lib.dram_conv3d_worklist(self._handle, _p(support), radius, _p(flags), _p(items), _p(count),
                                             _stream()), "dram_conv3d_worklist")

    def run_listed(self, items, count, max_ctas=0):
        """`run` restricted to the listed work items; the other output voxels keep their values."""
        check(self._lib.dram_conv3d_run_listed(self._handle, _p(items), _p(count), max_ctas, _stream()),
              "dram_conv3d_run_listed")
        return self.out

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h:
            try:
                self._lib.dram_conv3d_plan_destroy(h)
            except Exception:
                pass
            self._handle = None


def pow2_normalizer(w2d):
    """Per-row power of two m with max|row| / m in [0.5, 1): dividing by it is exact and keeps every
    packed weight in the normal range of fp16; the kernel multiplies the accumulator by m again."""
    amax = w2d.abs().amax(dim=1).clamp_min(2.0 ** -100)
    return torch.exp2(torch.floor(torch.log2(amax)) + 1.0)


def pack_conv_weight(weight, scale=None, dtype=torch.bfloat16, normalize=False):
    """[Cout, Cin, kd, kh, kw] fp32 -> 16-bit [Cout, kd*kh*kw*Cin] (tap-major, channel-minor).

    `scale` (fp32 [Cout]) is the folded BatchNorm factor gamma/sqrt(var+eps), multiplied in fp32
    before the single rounding to `dtype`.  With `normalize` the rows are divided by a power of two
    (exact) and `(packed, multiplier fp32 [Cout])` is returned for the epilogue `scale` argument.
    """
    w = weight.detach().to(torch.float32)
    if scale is not None:
        w = w * scale.to(torch.float32).view(-1, 1, 1, 1, 1)
    cout = w.shape[0]
    w = w.permute(0, 2, 3, 4, 1).reshape(cout, -1)
    if normalize:
        mult = pow2_normalizer(w)
        return (w / mult.view(-1, 1)).to(dtype).contiguous(), mult.contiguous()
    return w.to(dtype).contiguous()


def fold_bn(bn, conv_bias=None, eps=None):
    """Eval-mode BatchNorm3d as (scale, shift) fp32: y = conv*scale + shift."""
    eps = bn.eps if eps is None else eps
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + eps)
    shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
    if conv_bias is not None:
        shift = shift + conv_bias.detach().float() * scale
    return scale, shift


# --------------------------------------------------------------------------------------------
# stateless kernels
# --------------------------------------------------------------------------------------------
def stem_expand(x, out=None, dtype=torch.bfloat16):
    """fp32 [N, D, H, W] -> 16-bit [N, D, ceil(H/2), ceil(W/2), 64] (K2a)."""
    _need(x, torch.float32, "stem_expand x", 4)
    n, d, h, w = x.shape
    shape = (n, d, (h - 1) // 2 + 1, (w - 1) // 2 + 1, 64)
    if out is None:
        out = torch.empty(shape, dtype=dtype, device=x.device)
    _need16(out, "stem_expand out", 5)
    check(_capi.load().dram_stem_expand(_p(x), _p(out), n, d, h, w, ACT_DTYPES[out.dtype], _stream()),
          "dram_stem_expand")
    return out


def pack_stem_weight(weight, scale=None, dtype=torch.bfloat16, normalize=False):
    """conv1.weight [64, 1, 7, 7, 7] -> 16-bit [64, 7*64] matching `stem_expand` (k = kd*64 + kh*8 + kw)."""
    w = weight.detach().to(torch.float32)
    if scale is not None:
        w = w * scale.to(torch.float32).view(-1, 1, 1, 1, 1)
    cout = w.shape[0]
    packed = torch.zeros((cout, 7, 8, 8), dtype=torch.float32, device=w.device)
    packed[:, :, :7, :7] = w[:, 0]
    packed = packed.reshape(cout, 7 * 64)
    if normalize:
        mult = pow2_normalizer(packed)
        return (packed / mult.view(-1, 1)).to(dtype).contiguous(), mult.contiguous()
    return packed.to(dtype).contiguous()


def pack_stem_weight_fused(weight, scale=None, dtype=torch.bfloat16, normalize=False):
    """conv1.weight [64, 1, 7, 7, 7] -> the 16-bit operand of `stem_conv7`: 28672 values =
    even kd [kh=8][kd=6,4,2,0][cout=64][j=8] followed by odd kd [kh=8][kd=5,3,1][cout=64][j=8], element =
    w[cout, 0, kd, kh, j-1] (* scale[cout]) for kh < 7 and j >= 1, zero otherwise (the kernel's pseudo-channel j
    reads input column 2*ow - 4 + j; one input plane feeds the output planes of one kd parity with a single MMA).
    With `normalize` the per-output-channel power-of-two multiplier is returned as well (`pow2_normalizer`)."""
    w = weight.detach().to(torch.float32)
    if scale is not None:
        w = w * scale.to(torch.float32).view(-1, 1, 1, 1, 1)
    cout = w.shape[0]
    if tuple(w.shape) != (64, 1, 7, 7, 7):
        raise ValueError(f"pack_stem_weight_fused: expected conv1.weight [64,1,7,7,7], got {tuple(w.shape)}")
    mult = pow2_normalizer(w.reshape(cout, -1)) if normalize else None
    if normalize:
        w = w / mult.view(-1, 1, 1, 1, 1)
    full = torch.zeros((7, 8, cout, 8), dtype=torch.float32, device=w.device)   # [kd, kh, cout, j]
    full[:, :7, :, 1:] = w[:, 0].permute(1, 2, 0, 3)
    even = full[[6, 4, 2, 0]].permute(1, 0, 2, 3)   # [kh, 4, cout, j]
    odd = full[[5, 3, 1]].permute(1, 0, 2, 3)       # [kh, 3, cout, j]
    packed = torch.cat([even.reshape(-1), odd.reshape(-1)]).to(dtype).contiguous()
    return (packed, mult.contiguous()) if normalize else packed


def stem_conv7(x, weight, bias, scale=None, out=None, relu=True, max_ctas=0):
    """K2: fp32 [N, D, H, W] -> 16-bit NDHWC [N, D', H', W', 64] = relu(conv7^3 s2 p3 * scale + bias)."""
    lib = _capi.load()
    _need(x, torch.float32, "stem_conv7 x", 4)
    _need16(weight, "stem_conv7 weight", 1)
    if weight.numel() != 7 * 8 * 64 * 8:
        raise ValueError(f"stem_conv7: weight must hold 28672 values (pack_stem_weight_fused), got {tuple(weight.shape)}")
    _need(bias, torch.float32, "stem_conv7 bias", 1)
    if scale is not None:
        _need(scale, torch.float32, "stem_conv7 scale", 1)
    if bias.shape[0] != 64 or (scale is not None and scale.shape[0] != 64):
        raise ValueError("stem_conv7: bias/scale must have 64 entries")
    n, d, h, w = x.shape
    shape = (n, (d - 1) // 2 + 1, (h - 1) // 2 + 1, (w - 1) // 2 + 1, 64)
    if out is None:
        out = torch.empty(shape, dtype=weight.dtype, device=x.device)
    _need(out, weight.dtype, "stem_conv7 out", 5)
    if tuple(out.shape) != shape:
        raise ValueError(f"stem_conv7: out shape {tuple(out.shape)} != {shape}")
    check(lib.dram_stem_conv7(_p(x), _p(weight), _p(bias), _p(scale), _p(out), n, d, h, w, 1 if relu else 0,
                              ACT_DTYPES[weight.dtype], max_ctas, _stream()), "dram_stem_conv7")
    return out


def stem_conv7_hu(hu, lut, weight, bias, scale=None, out=None, relu=True, lo=-1150, max_ctas=0):
    """K2 fed from int16 HU [N, D, H, W] + the per-volume table fp32 [N, hi - lo + 1] of `window_lut`: window,
    standardise (K8's values, tabulated), conv 7^3 s2 p3, scale/shift, ReLU in one kernel; the fp32 image never exists."""
    lib = _capi.load()
    _need(hu, torch.int16, "stem_conv7_hu hu", 4)
    _need(lut, torch.float32, "stem_conv7_hu lut", 2)
    _need16(weight, "stem_conv7_hu weight", 1)
    if weight.numel() != 7 * 8 * 64 * 8:
        raise ValueError("stem_conv7_hu: weight must hold 28672 values (pack_stem_weight_fused)")
    _need(bias, torch.float32, "stem_conv7_hu bias", 1)
    if scale is not None:
        _need(scale, torch.float32, "stem_conv7_hu scale", 1)
    n, d, h, w = hu.shape
    if lut.shape[0] != n:
        raise ValueError(f"stem_conv7_hu: lut must have {n} rows, got {tuple(lut.shape)}")
    shape = (n, (d - 1) // 2 + 1, (h - 1) // 2 + 1, (w - 1) // 2 + 1, 64)
    if out is None:
        out = torch.empty(shape, dtype=weight.dtype, device=hu.device)
    _need(out, weight.dtype, "stem_conv7_hu out", 5)
    if tuple(out.shape) != shape:
        raise ValueError(f"stem_conv7_hu: out shape {tuple(out.shape)} != {shape}")
    check(lib.dram_stem_conv7_hu(_p(hu), _p(lut), int(lo), lut.shape[1], _p(weight), _p(bias), _p(scale), _p(out), n, d,
                                 h, w, 1 if relu else 0, ACT_DTYPES[weight.dtype], max_ctas, _stream()),
          "dram_stem_conv7_hu")
    return out


def maxpool3d(x, out=None):
    _need16(x, "maxpool3d x", 5)
    n, d, h, w, c = x.shape
    shape = (n, (d - 1) // 2 + 1, (h - 1) // 2 + 1, (w - 1) // 2 + 1, c)
    if out is None:
        out = torch.empty(shape, dtype=x.dtype, device=x.device)
    _need(out, x.dtype, "maxpool3d out", 5)
    check(_capi.load().dram_maxpool3d(_p(x), _p(out), n, d, h, w, c, ACT_DTYPES[x.dtype], _stream()),
          "dram_maxpool3d")
    return out


def upsample2x(x, out=None):
    _need16(x, "upsample2x x", 5)
    n, d, h, w, c = x.shape
    if out is None:
        out = torch.empty((n, 2 * d, 2 * h, 2 * w, c), dtype=x.dtype, device=x.device)
    _need(out, x.dtype, "upsample2x out", 5)
    check(_capi.load().dram_upsample2x(_p(x), _p(out), n, d, h, w, c, ACT_DTYPES[x.dtype], _stream()),
          "dram_upsample2x")
    return out


class Upsample2xPlan:
    """K4 on the tensor cores: x [N, D, H, W, C] (C % 64 == 0) -> out [N, 2D, 2H, 2W, C], fixed buffers."""

    def __init__(self, x, out=None):
        lib = _capi.load()
        _need16(x, "upsample2x x", 5)
        n, d, h, w, c = x.shape
        if out is None:
            out = torch.empty((n, 2 * d, 2 * h, 2 * w, c), dtype=x.dtype, device=x.device)
        _need(out, x.dtype, "upsample2x out", 5)
        if tuple(out.shape) != (n, 2 * d, 2 * h, 2 * w, c):
            raise ValueError(f"upsample2x: out shape {tuple(out.shape)} does not match x {tuple(x.shape)}")
        handle = C.c_void_p()
        check(lib.dram_upsample2x_plan_create(_p(x), _p(out), n, d, h, w, c, ACT_DTYPES[x.dtype], C.byref(handle)),
              "dram_upsample2x_plan_create")
        self._handle, self._lib, self._keep, self.out = handle, lib, (x, out), out

    def run(self, max_ctas=0):
        check(self._lib.dram_upsample2x_plan_run(self._handle, max_ctas, _stream()), "dram_upsample2x_plan_run")
        return self.out

    def worklist_size(self):
        n = C.c_int32()
        check(self._lib.dram_upsample2x_worklist_size(self._handle, C.byref(n)), "dram_upsample2x_worklist_size")
        return n.value

    def build_worklist(self, support, radius, flags, items, count):
        """As Conv3dPlan.build_worklist, over the 8x4x4 output bricks."""
        check(self._lib.dram_upsample2x_worklist(self._handle, _p(support), radius, _p(flags), _p(items), _p(count),
                                                 _stream()), "dram_upsample2x_worklist")

    def run_listed(self, items, count, max_ctas=0):
        check(self._lib.dram_upsample2x_plan_run_listed(self._handle, _p(items), _p(count), max_ctas, _stream()),
              "dram_upsample2x_plan_run_listed")
        return self.out

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h:
            try:
                self._lib.dram_upsample2x_plan_destroy(h)
            except Exception:
                pass
            self._handle = None


def decoder_support(ess, half_dims, rows=None, out=None):
    """The decoder-grid voxels K7 reads for `ess` uint8 [N, D, H, W]: bit mask int32 [N, d, h, ceil(w/32)] over the
    grid `half_dims` = (d, h, w) (see dram_decoder_support).  `rows` / `out`: optional preallocated scratch / result."""
    lib = _capi.load()
    _need(ess, torch.uint8, "decoder_support ess", 4)
    n, D, H, W = ess.shape
    d, h, w = half_dims
    words = (w + 31) // 32
    if rows is None:
        rows = torch.empty((n, D, H, words), dtype=torch.int32, device=ess.device)
    if out is None:
        out = torch.empty((n, d, h, words), dtype=torch.int32, device=ess.device)
    _need(rows, torch.int32, "decoder_support rows", 4)
    _need(out, torch.int32, "decoder_support out", 4)
    if tuple(rows.shape) != (n, D, H, words) or tuple(out.shape) != (n, d, h, words):
        raise ValueError("decoder_support: scratch / output shape mismatch")
    check(lib.dram_decoder_support(_p(ess), n, D, H, W, d, h, w, _p(rows), _p(out), _stream()), "dram_decoder_support")
    return out


def upconv_axis(x, axis, groups, out=None):
    """K13, one axis of the commuted up-sampled convolution.  x: 16-bit [N, d, h, w, C] whose first groups*192 channels
    are [groups][3 taps of `axis`][64]; returns [N, d', h', w', groups*64] with the size of `axis` (1 = D, 2 = H,
    3 = W) doubled: out[o] = sum_t lerp(x[.., t, :])(o + t - 1), zero outside (see include/dram_b200.h)."""
    _need16(x, "upconv_axis x", 5)
    if axis not in (1, 2, 3):
        raise ValueError("upconv_axis: axis must be 1 (D), 2 (H) or 3 (W)")
    n, d, h, w, c = x.shape
    if c < groups * 192:
        raise ValueError(f"upconv_axis: {c} channels cannot hold {groups} groups of 3 x 64")
    shape = [n, d, h, w, groups * 64]
    shape[axis] *= 2
    if out is None:
        out = torch.empty(shape, dtype=x.dtype, device=x.device)
    _need(out, x.dtype, "upconv_axis out", 5)
    if list(out.shape) != shape:
        raise ValueError(f"upconv_axis: out shape {tuple(out.shape)} != {tuple(shape)}")
    dims = (n, d, h, w)
    outer = 1
    for v in dims[:axis]:
        outer *= v
    inner = 1
    for v in dims[axis + 1:]:
        inner *= v
    check(_capi.load().dram_upconv_axis(_p(x), _p(out), outer, dims[axis], 2 * dims[axis], inner, groups, c,
                                        ACT_DTYPES[x.dtype], _stream()), "dram_upconv_axis")
    return out


def pack_upconv_weight(weight, c_up, scale=None, dtype=torch.bfloat16, pad_rows_to=256):
    """The up-sampled half of a decoder convolution [Cout=64, c_up + c_skip, 3, 3, 3] as the 1x1x1 operand of K13's
    low-resolution product: 16-bit [R, c_up], row tap*64 + co = weight[co, :c_up, tap] (* scale[co]), rows
    normalised by a power of two like `pack_conv_weight(normalize=True)`, R = 27*64 rounded up to `pad_rows_to` with
    zero rows; returns (packed, multiplier fp32 [R])."""
    w = weight.detach().to(torch.float32)[:, :c_up]
    if scale is not None:
        w = w * scale.to(torch.float32).view(-1, 1, 1, 1, 1)
    cout = w.shape[0]
    if cout != 64 or tuple(w.shape[2:]) != (3, 3, 3):
        raise ValueError(f"pack_upconv_weight: expected [64, C, 3, 3, 3], got {tuple(weight.shape)}")
    rows = w.reshape(cout, c_up, 27).permute(2, 0, 1).reshape(27 * cout, c_up)   # [tap][co] x ci
    mult = pow2_normalizer(rows)
    packed = (rows / mult.view(-1, 1)).to(dtype)
    if pad_rows_to > 1 and packed.shape[0] % pad_rows_to:
        # zero rows up to a multiple of the GEMM's N tile (27 * 64 = 1728 -> 1792 = 7 * 256); K13's W pass skips them
        extra = pad_rows_to - packed.shape[0] % pad_rows_to
        packed = torch.cat([packed, packed.new_zeros((extra, c_up))])
        mult = torch.cat([mult, mult.new_ones(extra)])
    return packed.contiguous(), mult.contiguous()


def masked_pool(dense, mask=None):
    """dense fp32 [N, C, d, h, w]; mask uint8 (binary) or fp32 (weights) [N, D, H, W] or None -> fp32 [N, C]."""
    lib = _capi.load()
    _need(dense, torch.float32, "masked_pool dense", 5)
    n, ch, d, h, w = dense.shape
    md = mh = mw = 0
    is_f32 = 0
    if mask is not None:
        is_f32 = 1 if mask.dtype == torch.float32 else 0
        _need(mask, torch.float32 if is_f32 else torch.uint8, "masked_pool mask", 4)
        if mask.shape[0] != n:
            raise ValueError("masked_pool: mask batch mismatch")
        md, mh, mw = mask.shape[1:]
    ws = torch.empty(lib.dram_pool_workspace_bytes(n, ch), dtype=torch.uint8, device=dense.device)
    out = torch.empty((n, ch), dtype=torch.float32, device=dense.device)
    check(lib.dram_masked_pool(_p(dense), _p(mask), is_f32, _p(out), _p(ws), n, ch, d, h, w, md, mh, mw, _stream()),
          "dram_masked_pool")
    return out


def dram_upsample_mask(dense0, dense1, ess, lungs, size, per_sample_denominator=False, out=None):
    """K7: returns (out0, out1 fp32 [N,1,D,H,W], pct fp32 [2, N]).  `out`: optional preallocated (out0, out1)."""
    lib = _capi.load()
    _need(dense0, torch.float32, "dram dense0", 5)
    _need(dense1, torch.float32, "dram dense1", 5)
    _need(ess, torch.uint8, "dram ess", 4)
    _need(lungs, torch.uint8, "dram lungs", 4)
    n, ch, d, h, w = dense0.shape
    if ch != 1 or dense1.shape != dense0.shape:
        raise ValueError("dram_upsample_mask: dense maps must be [N,1,d,h,w] and alike")
    D, H, W = size
    if tuple(ess.shape) != (n, D, H, W) or tuple(lungs.shape) != (n, D, H, W):
        raise ValueError("dram_upsample_mask: mask shape mismatch")
    if out is None:
        out0 = torch.empty((n, 1, D, H, W), dtype=torch.float32, device=dense0.device)
        out1 = torch.empty_like(out0)
    else:
        out0, out1 = out
        _need(out0, torch.float32, "dram out0", 5)
        _need(out1, torch.float32, "dram out1", 5)
        if tuple(out0.shape) != (n, 1, D, H, W) or tuple(out1.shape) != (n, 1, D, H, W):
            raise ValueError("dram_upsample_mask: out tensors must be [N,1,D,H,W]")
    pct = torch.empty((2, n), dtype=torch.float32, device=dense0.device)
    ws = torch.empty(lib.dram_dram_workspace_bytes(n), dtype=torch.uint8, device=dense0.device)
    check(lib.dram_dram_upsample_mask(_p(dense0), _p(dense1), _p(ess), _p(lungs), _p(out0), _p(out1), _p(pct),
                                      _p(ws), n, d, h, w, D, H, W, 1 if per_sample_denominator else 0,
                                      _stream()), "dram_dram_upsample_mask")
    return out0, out1, pct


LOBE_LABELS = 256


def lobe_scores(cle, pse, ess, labels, out=None):
    """K7l: lesion percentages per label.  cle, pse fp32 [B,1,D,H,W] (the dRAM maps of K7); ess bool or uint8 and
    labels uint8, both [B,D,H,W].  Returns (pct fp32 [2, B, 256], voxels int64 [B, 256]): voxels[b, k] counts the
    voxels labelled k; pct[m, b, k] is the sum of map m over the ess voxels labelled k divided by voxels[b, k] (NaN
    where that is 0).  `out`: optional preallocated (pct, voxels)."""
    lib = _capi.load()
    _need(cle, torch.float32, "lobe_scores cle", 5)
    _need(pse, torch.float32, "lobe_scores pse", 5)
    if isinstance(ess, torch.Tensor) and ess.dtype == torch.bool:
        ess = ess.view(torch.uint8)
    _need(ess, torch.uint8, "lobe_scores ess", 4)
    _need(labels, torch.uint8, "lobe_scores labels", 4)
    B, D, H, W = labels.shape
    if tuple(cle.shape) != (B, 1, D, H, W) or tuple(pse.shape) != (B, 1, D, H, W) or tuple(ess.shape) != (B, D, H, W):
        raise ValueError(f"lobe_scores: maps {tuple(cle.shape)} / {tuple(pse.shape)} and ess {tuple(ess.shape)} must "
                         f"match labels {tuple(labels.shape)}")
    if out is None:
        pct = torch.empty((2, B, LOBE_LABELS), dtype=torch.float32, device=labels.device)
        voxels = torch.empty((B, LOBE_LABELS), dtype=torch.int64, device=labels.device)
    else:
        pct, voxels = out
        _need(pct, torch.float32, "lobe_scores out pct", 3)
        _need(voxels, torch.int64, "lobe_scores out voxels", 2)
        if tuple(pct.shape) != (2, B, LOBE_LABELS) or tuple(voxels.shape) != (B, LOBE_LABELS):
            raise ValueError(f"lobe_scores: out must be ([2, {B}, 256], [{B}, 256])")
    count = D * H * W
    ws = torch.empty(lib.dram_lobe_workspace_bytes(B, count) // 8, dtype=torch.float64, device=labels.device)
    check(lib.dram_lobe_sums(_p(cle), _p(pse), _p(ess), _p(labels), _p(pct), _p(voxels), _p(ws), B, count, _stream()),
          "dram_lobe_sums")
    return pct, voxels


def window_standardize(hu, lo=-1150.0, hi=-300.0, out=None, batched=False):
    """K8: int16 HU -> fp32 standardised window; returns (out, stats).  One volume of any shape (stats fp32 [2]),
    or with `batched` a stack [N, ...] of volumes with per-volume statistics (stats fp32 [N, 2]) in three launches."""
    lib = _capi.load()
    _need(hu, torch.int16, "window_standardize hu")
    n = hu.shape[0] if batched else 1
    if out is None:
        out = torch.empty(hu.shape, dtype=torch.float32, device=hu.device)
    _need(out, torch.float32, "window_standardize out")
    stats = torch.empty((n, 2) if batched else (2,), dtype=torch.float32, device=hu.device)
    ws = torch.empty(lib.dram_preprocess_workspace_bytes_n(n) // 8, dtype=torch.float64, device=hu.device)
    check(lib.dram_window_standardize_batch(_p(hu), _p(out), _p(stats), _p(ws), n, hu.numel() // n, lo, hi, _stream()),
          "dram_window_standardize")
    return out, stats


def window_stats(hu, lo=-1150.0, hi=-300.0):
    """K8, statistics pass only: int16 HU [N, ...] -> fp32 [N, 2] = (mean, unbiased std) of each windowed volume."""
    lib = _capi.load()
    _need(hu, torch.int16, "window_stats hu")
    n = hu.shape[0]
    stats = torch.empty((n, 2), dtype=torch.float32, device=hu.device)
    ws = torch.empty(lib.dram_preprocess_workspace_bytes_n(n) // 8, dtype=torch.float64, device=hu.device)
    check(lib.dram_window_stats(_p(hu), _p(stats), _p(ws), n, hu.numel() // n, lo, hi, _stream()), "dram_window_stats")
    return stats


def window_lut(hu, lo=-1150, hi=-300):
    """K8 as a table: int16 HU [N, ...] -> (lut fp32 [N, hi - lo + 1], stats fp32 [N, 2]); lut[v, i] is the value
    `window_standardize` gives a voxel of HU lo + i of volume v (voxels outside the window clamp to its ends)."""
    lib = _capi.load()
    _need(hu, torch.int16, "window_lut hu")
    if int(lo) != lo or int(hi) != hi:
        raise ValueError("window_lut: the window bounds must be integers")
    n = hu.shape[0]
    lut = torch.empty((n, int(hi) - int(lo) + 1), dtype=torch.float32, device=hu.device)
    stats = torch.empty((n, 2), dtype=torch.float32, device=hu.device)
    ws = torch.empty(lib.dram_preprocess_workspace_bytes_n(n) // 8, dtype=torch.float64, device=hu.device)
    check(lib.dram_window_lut(_p(hu), _p(lut), _p(stats), _p(ws), n, hu.numel() // n, float(lo), float(hi), _stream()),
          "dram_window_lut")
    return lut, stats


def slice_index(d_in, d_out, device):
    """The D-slice pick of Interpolate (spatial_transforms.py:66), built with the same torch ops."""
    return torch.linspace(0, d_in - 1, d_out).long().to(torch.int32).to(device)


def resize_image(x, size):
    _need(x, torch.float32, "resize_image x", 3)
    D, H, W = x.shape
    D2, H2, W2 = size
    idx = slice_index(D, D2, x.device)
    out = torch.empty((D2, H2, W2), dtype=torch.float32, device=x.device)
    check(_capi.load().dram_resize_image(_p(x), _p(out), _p(idx), D, H, W, D2, H2, W2, _stream()),
          "dram_resize_image")
    return out


def resize_mask(x, size):
    _need(x, torch.uint8, "resize_mask x", 3)
    D, H, W = x.shape
    D2, H2, W2 = size
    idx = slice_index(D, D2, x.device)
    out = torch.empty((D2, H2, W2), dtype=torch.uint8, device=x.device)
    check(_capi.load().dram_resize_mask(_p(x), _p(out), _p(idx), D, H, W, D2, H2, W2, _stream()),
          "dram_resize_mask")
    return out


def resize_labels(x, size, out=None):
    """uint8 label volume [D,H,W] -> `size`: the voxel `resize_mask` picks, its value kept (not cast to 0/1)."""
    _need(x, torch.uint8, "resize_labels x", 3)
    D, H, W = x.shape
    D2, H2, W2 = size
    idx = slice_index(D, D2, x.device)
    if out is None:
        out = torch.empty((D2, H2, W2), dtype=torch.uint8, device=x.device)
    _need(out, torch.uint8, "resize_labels out", 3)
    if tuple(out.shape) != (D2, H2, W2):
        raise ValueError(f"resize_labels: out shape {tuple(out.shape)} != {(D2, H2, W2)}")
    check(_capi.load().dram_resize_labels(_p(x), _p(out), _p(idx), D, H, W, D2, H2, W2, _stream()),
          "dram_resize_labels")
    return out


def mask_bbox(mask):
    """f1: uint8 [D,H,W] device mask -> int32[6] device tensor {zmin, zmax+1, ymin, ymax+1, xmin, xmax+1}
    of mask != 0 ({D,0,H,0,W,0} when the mask is empty)."""
    _need(mask, torch.uint8, "mask_bbox mask", 3)
    D, H, W = mask.shape
    bbox = torch.empty(6, dtype=torch.int32, device=mask.device)
    check(_capi.load().dram_mask_bbox(_p(mask), D, H, W, _p(bbox), _stream()), "dram_mask_bbox")
    return bbox


def lung_crop(scan, lobe, crop, out=None):
    """f1 (dataset.py:66-80): int16 scan + uint8 lobe labels [D,H,W] and crop ((z0,z1),(y0,y1),(x0,x1)) ->
    (image int16, lung uint8, ess uint8) of the crop size: blanking outside the twice-dilated lung, LAA-910.
    `out`: optional preallocated (image, lung, ess) of the crop size (e.g. slices of a batch buffer)."""
    lib = _capi.load()
    _need(scan, torch.int16, "lung_crop scan", 3)
    _need(lobe, torch.uint8, "lung_crop lobe", 3)
    if scan.shape != lobe.shape:
        raise ValueError("scan and lobe segmentation have different shapes.")
    D, H, W = scan.shape
    (z0, z1), (y0, y1), (x0, x1) = [(int(a), int(b)) for a, b in crop]
    cd, ch, cw = z1 - z0, y1 - y0, x1 - x0
    if out is None:
        image = torch.empty((cd, ch, cw), dtype=torch.int16, device=scan.device)
        lung = torch.empty((cd, ch, cw), dtype=torch.uint8, device=scan.device)
        ess = torch.empty_like(lung)
    else:
        image, lung, ess = out
        _need(image, torch.int16, "lung_crop out image", 3)
        _need(lung, torch.uint8, "lung_crop out lung", 3)
        _need(ess, torch.uint8, "lung_crop out ess", 3)
        if not (tuple(image.shape) == tuple(lung.shape) == tuple(ess.shape) == (cd, ch, cw)):
            raise ValueError(f"lung_crop: out tensors must have the crop shape {(cd, ch, cw)}")
    ws = torch.empty(lib.dram_lung_crop_workspace_bytes(cd, ch, cw), dtype=torch.uint8, device=scan.device)
    check(lib.dram_lung_crop(_p(scan), _p(lobe), D, H, W, z0, y0, x0, cd, ch, cw, _p(image), _p(lung), _p(ess),
                             _p(ws), _stream()), "dram_lung_crop")
    return image, lung, ess


HU_BINS = 2048      # HU histogram bins: bin b holds HU b - 1024 (values clamped to [-1024, 1023])
HU_SLOTS = 16       # labels per histogram pass


def label_counts(labels):
    """Voxels per label of a uint8 label volume (any shape): int64 [256] on the device, exact."""
    _need(labels, torch.uint8, "label_counts labels")
    counts = torch.empty(LOBE_LABELS, dtype=torch.int64, device=labels.device)
    check(_capi.load().dram_label_counts(_p(labels), labels.numel(), _p(counts), _stream()), "dram_label_counts")
    return counts


def hu_histograms(scan, labels, label_ids):
    """HU histograms of the voxels of each label in `label_ids` (distinct ints in 0..255): int16 scan and uint8 labels
    of one shape.  Returns (hist int64 [len(ids), 2048], hu_sum int64 [len(ids)]) on the device: hist[i, b] counts
    the voxels labelled label_ids[i] whose HU, clamped to [-1024, 1023], is b - 1024; hu_sum[i] is the exact sum of
    their unclamped HU.  One pass per group of 16 labels; no host synchronisation."""
    lib = _capi.load()
    _need(scan, torch.int16, "hu_histograms scan")
    _need(labels, torch.uint8, "hu_histograms labels")
    if scan.shape != labels.shape:
        raise ValueError(f"hu_histograms: scan {tuple(scan.shape)} and labels {tuple(labels.shape)} differ in shape")
    ids = [int(k) for k in label_ids]
    if any(not 0 <= k < LOBE_LABELS for k in ids) or len(set(ids)) != len(ids):
        raise ValueError(f"hu_histograms: label ids must be distinct values in 0..255, got {ids}")
    hist = torch.empty((len(ids), HU_BINS), dtype=torch.int64, device=scan.device)
    hu_sum = torch.empty(len(ids), dtype=torch.int64, device=scan.device)
    for g in range(0, len(ids), HU_SLOTS):
        group = ids[g:g + HU_SLOTS]
        table = bytearray(b"\xff" * LOBE_LABELS)
        for s, k in enumerate(group):
            table[k] = s
        check(lib.dram_label_hu_hist(_p(scan), _p(labels), scan.numel(), bytes(table), len(group), _p(hist[g:]),
                                     _p(hu_sum[g:]), _stream()), "dram_label_hu_hist")
    return hist, hu_sum


def heatmap_u8(dram_map, crop, original_size, out=None):
    """f2 (processor.py:111-158): one fp32 dRAM [d,h,w] -> uint8 [D,H,W] of the original scan: trilinear
    (align_corners) to the crop size, pasted at `crop`, windowed (0,1)->(0,255) with truncation."""
    _need(dram_map, torch.float32, "heatmap_u8 map", 3)
    d, h, w = dram_map.shape
    OD, OH, OW = (int(v) for v in original_size)
    (z0, z1), (y0, y1), (x0, x1) = [(int(a), int(b)) for a, b in crop]
    if out is None:
        out = torch.empty((OD, OH, OW), dtype=torch.uint8, device=dram_map.device)
    _need(out, torch.uint8, "heatmap_u8 out", 3)
    check(_capi.load().dram_heatmap_u8(_p(dram_map), d, h, w, _p(out), OD, OH, OW, z0, y0, x0, z1 - z0, y1 - y0,
                                       x1 - x0, _stream()), "dram_heatmap_u8")
    return out


def to_ndhwc_16(x, dtype=torch.bfloat16):
    """fp32 NCDHW -> 16-bit NDHWC."""
    _need(x, torch.float32, "to_ndhwc_16 x", 5)
    n, c, d, h, w = x.shape
    out = torch.empty((n, d, h, w, c), dtype=dtype, device=x.device)
    check(_capi.load().dram_ncdhw_f32_to_ndhwc_16(_p(x), _p(out), n, c, d, h, w, ACT_DTYPES[dtype], _stream()),
          "dram_ncdhw_f32_to_ndhwc_16")
    return out


def to_ndhwc_bf16(x):
    return to_ndhwc_16(x, torch.bfloat16)


def to_ncdhw_f32(x):
    """16-bit NDHWC -> fp32 NCDHW."""
    _need16(x, "to_ncdhw_f32 x", 5)
    n, d, h, w, c = x.shape
    out = torch.empty((n, c, d, h, w), dtype=torch.float32, device=x.device)
    check(_capi.load().dram_ndhwc_16_to_ncdhw_f32(_p(x), _p(out), n, c, d, h, w, ACT_DTYPES[x.dtype], _stream()),
          "dram_ndhwc_16_to_ncdhw_f32")
    return out


from . import custom_ops  # noqa: E402,F401  (registers the dram_b200:: torch.library operators)
