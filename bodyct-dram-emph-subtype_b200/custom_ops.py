"""`torch.library` registration of the C-ABI kernels: the `dram_b200::` operator namespace.

Every stateless kernel family of libdram_b200.so is a `torch.library.custom_op` here (CUDA implementation =
the ctypes wrapper in `ops.py`; fake/meta implementation = shape inference only), so the kernels

  * appear under their own names in `torch.profiler` traces and `torch.ops.dram_b200.*`,
  * can be traced with FakeTensors / `torch.compile(fullgraph=True)` around them and pass `torch.library.opcheck`,
  * capture into CUDA graphs like any ATen op (they launch on `torch.cuda.current_stream()`, allocate through the
    caching allocator only and never synchronise).

`dram_b200::conv3d` is the functional form of K1: it builds the TMA tensor maps for the tensors it is given, launches
and drops the plan (the maps travel to the kernel by value as `__grid_constant__` parameters).  The network itself does
not go through the dispatcher: `engine.Med3DEngine` keeps frozen `ops.Conv3dPlan`s over address-stable buffers and
replays them as ONE CUDA graph, which is cheaper than ~50 dispatcher calls per volume.

There is no CPU implementation: calling an op with CPU tensors raises (NotImplementedError from the dispatcher).
"""
from typing import List, Optional, Tuple

import torch
from torch.library import custom_op

from . import ops

NS = "dram_b200"


def _half_up(n):
    return (n - 1) // 2 + 1


# ------------------------------------------------------------------------------------------------ K1
@custom_op(f"{NS}::conv3d", mutates_args=(), device_types="cuda")
def conv3d(x1: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, x2: Optional[torch.Tensor] = None,
           scale: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None, kernel: int = 3,
           stride: int = 1, dilation: int = 1, relu: bool = True, res_stride: int = 1) -> torch.Tensor:
    """NDHWC 16-bit conv3d (+ second K source, + per-channel scale/shift, + residual incl. shortcut A, + ReLU):
    nn.Conv3d + BatchNorm3d(eval) + ReLU + `out += residual` of med3d.py:93-184 in one launch.  `weight` is the packed
    [Cout, taps * (C1 + C2)] matrix of `ops.pack_conv_weight`; padding = dilation * (kernel - 1) / 2 ("same")."""
    plan = ops.Conv3dPlan(x1, weight, bias, x2=x2, scale=scale, kernel=kernel, stride=stride, dilation=dilation,
                          relu=relu, residual=residual, res_stride=res_stride)
    return plan.run()


@conv3d.register_fake
def _(x1, weight, bias, x2=None, scale=None, residual=None, kernel=3, stride=1, dilation=1, relu=True, res_stride=1):
    n, d, h, w, _ = x1.shape
    pad = dilation * (kernel - 1) // 2
    o = [(v + 2 * pad - dilation * (kernel - 1) - 1) // stride + 1 for v in (d, h, w)]
    return x1.new_empty((n, o[0], o[1], o[2], weight.shape[0]))


# ------------------------------------------------------------------------------------------------ K2
@custom_op(f"{NS}::stem_conv7", mutates_args=(), device_types="cuda")
def stem_conv7(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, scale: Optional[torch.Tensor] = None,
               relu: bool = True) -> torch.Tensor:
    """conv1 (7^3, stride 2, pad 3, 1 -> 64) + bn1 + ReLU from the fp32 image (med3d.py:296-304, 371-373)."""
    return ops.stem_conv7(x, weight, bias, scale, relu=relu)


@stem_conv7.register_fake
def _(x, weight, bias, scale=None, relu=True):
    n, d, h, w = x.shape
    return weight.new_empty((n, _half_up(d), _half_up(h), _half_up(w), 64))


# ------------------------------------------------------------------------------------------------ K3 / K4
@custom_op(f"{NS}::maxpool3d", mutates_args=(), device_types="cuda")
def maxpool3d(x: torch.Tensor) -> torch.Tensor:
    """MaxPool3d(3, stride 2, pad 1) on NDHWC 16-bit (med3d.py:305)."""
    return ops.maxpool3d(x)


@maxpool3d.register_fake
def _(x):
    n, d, h, w, c = x.shape
    return x.new_empty((n, _half_up(d), _half_up(h), _half_up(w), c))


@custom_op(f"{NS}::upsample2x", mutates_args=(), device_types="cuda")
def upsample2x(x: torch.Tensor) -> torch.Tensor:
    """Upsample(scale 2, trilinear, align_corners=True) on NDHWC 16-bit (med3d.py:83, 86)."""
    return ops.upsample2x(x)


@upsample2x.register_fake
def _(x):
    n, d, h, w, c = x.shape
    return x.new_empty((n, 2 * d, 2 * h, 2 * w, c))


# ------------------------------------------------------------------------------------------------ K6 / K7
@custom_op(f"{NS}::masked_pool", mutates_args=(), device_types="cuda")
def masked_pool(dense: torch.Tensor, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Lobe-masked (mask given: nearest-resized to the map, med3d.py:383-387) or global (med3d.py:284) mean."""
    return ops.masked_pool(dense, mask)


@masked_pool.register_fake
def _(dense, mask=None):
    return dense.new_empty((dense.shape[0], dense.shape[1]))


@custom_op(f"{NS}::dram_upsample_mask", mutates_args=(), device_types="cuda")
def dram_upsample_mask(dense0: torch.Tensor, dense1: torch.Tensor, ess: torch.Tensor, lungs: torch.Tensor,
                       per_sample_denominator: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """dRAM of models.py:438-441: both maps trilinear (align_corners) to the size of `ess`, times `ess`, and the
    lesion percentages over the batch's (or each sample's) lung volume."""
    return ops.dram_upsample_mask(dense0, dense1, ess, lungs, tuple(ess.shape[1:]),
                                  per_sample_denominator=per_sample_denominator)


@dram_upsample_mask.register_fake
def _(dense0, dense1, ess, lungs, per_sample_denominator=False):
    n, D, H, W = ess.shape
    return (dense0.new_empty((n, 1, D, H, W)), dense0.new_empty((n, 1, D, H, W)), dense0.new_empty((2, n)))


@custom_op(f"{NS}::lobe_scores", mutates_args=(), device_types="cuda")
def lobe_scores(cle: torch.Tensor, pse: torch.Tensor, ess: torch.Tensor,
                labels: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Lesion percentages of both dRAM maps per label of a uint8 label volume (per lobe): (pct fp32 [2, B, 256],
    voxels int64 [B, 256]), each label divided by its own voxel count."""
    return ops.lobe_scores(cle, pse, ess, labels)


@lobe_scores.register_fake
def _(cle, pse, ess, labels):
    B = labels.shape[0]
    return (cle.new_empty((2, B, ops.LOBE_LABELS)), cle.new_empty((B, ops.LOBE_LABELS), dtype=torch.int64))


# ------------------------------------------------------------------------------------------------ K8 / K8b
@custom_op(f"{NS}::window_standardize", mutates_args=(), device_types="cuda")
def window_standardize(hu: torch.Tensor, lo: float = -1150.0, hi: float = -300.0) -> Tuple[torch.Tensor, torch.Tensor]:
    """IntensityWindow + Standardize of one int16 HU volume (functional.py:13-26, intensity_transforms.py:104-114);
    returns (fp32 volume, [mean, unbiased std])."""
    return ops.window_standardize(hu, lo, hi)


@window_standardize.register_fake
def _(hu, lo=-1150.0, hi=-300.0):
    return hu.new_empty(hu.shape, dtype=torch.float32), hu.new_empty((2,), dtype=torch.float32)


@custom_op(f"{NS}::resize_image", mutates_args=(), device_types="cuda")
def resize_image(x: torch.Tensor, size: List[int]) -> torch.Tensor:
    """Interpolate transform, image branch (spatial_transforms.py:55-75)."""
    return ops.resize_image(x, tuple(size))


@resize_image.register_fake
def _(x, size):
    return x.new_empty(tuple(size))


@custom_op(f"{NS}::resize_mask", mutates_args=(), device_types="cuda")
def resize_mask(x: torch.Tensor, size: List[int]) -> torch.Tensor:
    """Interpolate transform, mask branch (spatial_transforms.py:77-97)."""
    return ops.resize_mask(x, tuple(size))


@resize_mask.register_fake
def _(x, size):
    return x.new_empty(tuple(size))


# ------------------------------------------------------------------------------------------------ f2
@custom_op(f"{NS}::heatmap_u8", mutates_args=(), device_types="cuda")
def heatmap_u8(dram_map: torch.Tensor, crop: List[int], original_size: List[int]) -> torch.Tensor:
    """processor.py:111-158 for one map: resample to the crop box (z0, z1, y0, y1, x0, x1), paste, window to uint8."""
    box = [(crop[0], crop[1]), (crop[2], crop[3]), (crop[4], crop[5])]
    return ops.heatmap_u8(dram_map, box, tuple(original_size))


@heatmap_u8.register_fake
def _(dram_map, crop, original_size):
    return dram_map.new_empty(tuple(original_size), dtype=torch.uint8)


# ------------------------------------------------------------------------------------------------ densitometry
@custom_op(f"{NS}::label_counts", mutates_args=(), device_types="cuda")
def label_counts(labels: torch.Tensor) -> torch.Tensor:
    """Voxels per label of a uint8 label volume: int64 [256]."""
    return ops.label_counts(labels)


@label_counts.register_fake
def _(labels):
    return labels.new_empty((ops.LOBE_LABELS,), dtype=torch.int64)


@custom_op(f"{NS}::hu_histograms", mutates_args=(), device_types="cuda")
def hu_histograms(scan: torch.Tensor, labels: torch.Tensor, label_ids: List[int]) -> Tuple[torch.Tensor, torch.Tensor]:
    """HU histograms (clamped to [-1024, 1023], 2048 bins) and exact HU sums of the voxels of each listed label:
    (int64 [len(ids), 2048], int64 [len(ids)])."""
    return ops.hu_histograms(scan, labels, label_ids)


@hu_histograms.register_fake
def _(scan, labels, label_ids):
    n = len(label_ids)
    return scan.new_empty((n, ops.HU_BINS), dtype=torch.int64), scan.new_empty((n,), dtype=torch.int64)


REGISTERED = ("conv3d", "stem_conv7", "maxpool3d", "upsample2x", "masked_pool", "dram_upsample_mask",
              "window_standardize", "resize_image", "resize_mask", "heatmap_u8", "lobe_scores", "label_counts",
              "hu_histograms")
