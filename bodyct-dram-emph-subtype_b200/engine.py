"""Static execution plan of one Med3D seg-reg / seg-cls forward on one B200.

For a fixed (batch, D, H, W) the planner folds eval-mode BatchNorm into bf16 weights, lays out every
activation as NDHWC bf16 in HBM, builds one `Conv3dPlan` (TMA tensor maps + tile geometry) per
convolution and records the launch sequence.  `run()` replays it on the current CUDA stream; nothing
is allocated and no host<->device synchronisation happens after the plan exists.

Data flow (reference: med3d.py:369-388 / 270-285), all kernels from libdram_b200.so:
    image fp32 --K2a stem_expand--> 64 pseudo-channels --K1(7x1x1,s2)--> x (64ch, /2)
    x --K3 maxpool--> xp (/4) --K1 blocks layer1..4--> x1 (/4), x4 (/8, dilated)
    x4 --K4 up2x--> up1;  K1([up1 | x1]) -> K1 -> xup1 (/4)
    xup1 --K4 up2x--> up2; K1([up2 | x]) -> K1 -> xup2 (/2)
    xup2 --K1(64->32)+heads(+sigmoid) in the epilogue--> dense maps fp32 NCDHW (xup3 never stored)
    dense (+ lungs) --K6 masked/global pooling--> scores
"""
import os

import torch

from . import ops

LAYER_CFG = ((64, 1, 1), (128, 2, 1), (256, 1, 2), (512, 1, 4))  # planes, stride, dilation


def _conv_out(n, k, s, d, p):
    return (n + 2 * p - d * (k - 1) - 1) // s + 1


class _Step:
    """One launch of the recorded sequence."""

    __slots__ = ("name", "fn", "flops", "executed_flops", "conv_part")

    def __init__(self, name, fn, flops=0, executed_flops=None, conv_part=False):
        self.name, self.fn, self.flops = name, fn, flops
        self.executed_flops = flops if executed_flops is None else executed_flops
        # launches without FLOPs of their own that belong to a convolution's time (K13's interpolation passes)
        self.conv_part = conv_part or flops > 0


class Med3DEngine:
    def __init__(self, model, batch, dims, device, act_dtype=None):
        if device.type != "cuda":
            raise RuntimeError("Med3DEngine needs a CUDA device: this path has no CPU implementation")
        self.model = model
        self.act_dtype = ops.default_act_dtype() if act_dtype is None else act_dtype
        self.batch, self.dims, self.device = batch, tuple(dims), device
        self.head_kind = model.head_kind
        self._weights = {}    # name -> (packed weight bf16, bias fp32) device buffers (stable addresses)
        self._packers = []    # closures that (re)fill the buffers from the module's parameters
        self.steps = []
        self.conv_flops = 0
        self._graph = None
        self._graph_restricted = None
        self._restricted = None   # (support scratch, support bits, launch list) of run_network(active_ess=...)
        self._sat_counter = torch.zeros(1, dtype=torch.int32, device=device)
        self._sat_checked_epoch = None
        self.last_saturation_count = None   # result of the latest probed pass (None: never probed)
        self._build()
        self._weights_epoch = model.weights_epoch

    # ---------------------------------------------------------------- weights
    # The packed operands follow the module's parameters through `model.weights_epoch`, a counter the module bumps
    # in load_state_dict / _apply / train<->eval transitions / mark_weights_changed() (med3d._Med3DSegNet); run()
    # compares two integers.  (Round 1 hashed every parameter's version counter per run: 0.65 ms of host time.)

    def _register_weight(self, name, pack_fn):
        """pack_fn() -> (16-bit [cout, K], fp32 bias [cout], fp32 multiplier [cout]) on self.device;
        the buffers are refilled in place so the tensor maps built on them stay valid."""
        bufs = tuple(t.to(self.device).contiguous() for t in pack_fn())
        self._weights[name] = bufs

        def refill(bufs=bufs, pack_fn=pack_fn):
            for dst, src in zip(bufs, pack_fn()):
                dst.copy_(src)

        self._packers.append(refill)
        return bufs

    def refresh_weights(self):
        """Re-folds BatchNorm and re-packs every weight in place (after load_state_dict etc.)."""
        for refill in self._packers:
            refill()
        self._weights_epoch = self.model.weights_epoch

    def _conv_bn(self, name, conv, bn, stem=False):
        def pack():
            scale, shift = ops.fold_bn(bn, conv.bias)
            w = conv.weight.detach().to(self.device)
            fn = ops.pack_stem_weight if stem else ops.pack_conv_weight
            packed, mult = fn(w, scale.to(self.device), dtype=self.act_dtype, normalize=True)
            return packed, shift.to(self.device).float(), mult

        return self._register_weight(name, pack)

    # ---------------------------------------------------------------- plan
    def _add_conv(self, name, x1, wb, *, x2=None, kernel=3, stride=1, dilation=1, padding=None, relu=True,
                  residual=None, res_stride=1, heads=None, store_out=True, tile=None, flops=None,
                  upsample_x1=False, epilogue="auto"):
        plan = ops.Conv3dPlan(x1, wb[0], wb[1], x2=x2, scale=wb[2], kernel=kernel, stride=stride, dilation=dilation,
                              padding=padding, relu=relu, residual=residual, res_stride=res_stride,
                              heads=heads, store_out=store_out, tile=tile, upsample_x1=upsample_x1, epilogue=epilogue)
        fl = plan.flops if flops is None else flops
        self.conv_flops += fl
        self.steps.append(_Step(name, plan.run, fl, plan.executed_flops))
        return plan

    def _build(self):
        m, dev, B = self.model, self.device, self.batch
        D, H, W = self.dims
        e = m.expansion
        bf = self.act_dtype
        D1, H1, W1 = (_conv_out(n, 7, 2, 1, 3) for n in (D, H, W))
        D2, H2, W2 = (_conv_out(n, 3, 2, 1, 1) for n in (D1, H1, W1))
        D3, H3, W3 = (_conv_out(n, 3, 2, 1, 1) for n in (D2, H2, W2))
        if (2 * D3, 2 * H3, 2 * W3) != (D2, H2, W2) or (2 * D2, 2 * H2, 2 * W2) != (D1, H1, W1):
            # 2*ceil(n/2) >= n: the x2 up-sampled map is never SMALLER than its skip tensor, so the centre crop of
            # crop_concat_5d (med3d.py:39-48) is always the identity and a mismatch means "larger" — where the
            # reference's torch.cat fails with a size error as well
            raise ValueError(
                f"input size {self.dims}: each of D, H, W must be 8k or 8k-1 so that the x2 up-sampled maps match "
                "their skip tensors (the reference's crop_concat_5d/torch.cat raises for other sizes too)")
        # ---- stem: conv(7^3, s2, p3) + BN + ReLU straight from the fp32 image (K2); the older two-kernel
        # route (K2a unfold + K1 7x1x1) stays selectable for A/B runs with DRAM_B200_STEM=unfold
        self.image = torch.empty((B, D, H, W), dtype=torch.float32, device=dev)
        stem_flops = 2 * B * D1 * H1 * W1 * 64 * 343
        if os.environ.get("DRAM_B200_STEM", "fused").lower() == "unfold":
            self.xe = torch.empty((B, D, H1, W1, 64), dtype=bf, device=dev)
            self.steps.append(_Step("stem_expand", lambda: ops.stem_expand(self.image, out=self.xe)))
            wb = self._conv_bn("conv1", m.conv1, m.bn1, stem=True)
            x = self._add_conv("conv1", self.xe, wb, kernel=(7, 1, 1), stride=(2, 1, 1), padding=(3, 0, 0),
                               tile=(16, 8, 1), flops=stem_flops).out
        else:
            def pack_stem():
                scale, shift = ops.fold_bn(m.bn1, m.conv1.bias)
                packed, mult = ops.pack_stem_weight_fused(m.conv1.weight.detach().to(dev), scale.to(dev),
                                                          dtype=bf, normalize=True)
                return packed, shift.to(dev).float(), mult

            sw = self._register_weight("conv1", pack_stem)
            x = torch.empty((B, D1, H1, W1, 64), dtype=bf, device=dev)
            self.stem_weights, self.stem_out = sw, x   # for the int16-HU stem (predict_step_from_hu)
            self.conv_flops += stem_flops
            # the fused stem pads K from 343 to 7 * 8 * 8 = 448 and its tiles to 8 x 16 x 4 output voxels
            cd = lambda a, b: -(-a // b)  # noqa: E731
            stem_exec = 2 * B * (cd(D1, 4) * 4) * (cd(H1, 16) * 16) * (cd(W1, 8) * 8) * 64 * 448
            self.steps.append(_Step("conv1", lambda: ops.stem_conv7(self.image, sw[0], sw[1], sw[2], out=x),
                                    stem_flops, stem_exec))
        # ---- maxpool
        self.xp = torch.empty((B, D2, H2, W2, 64), dtype=bf, device=dev)
        self.steps.append(_Step("maxpool", lambda x=x: ops.maxpool3d(x, out=self.xp)))
        # ---- residual layers
        cur, inplanes = self.xp, 64
        feats = []
        for li, ((planes, stride, dil), layer) in enumerate(zip(LAYER_CFG, (m.layer1, m.layer2, m.layer3, m.layer4)), 1):
            for bi, blk in enumerate(layer):
                s = stride if bi == 0 else 1
                name = f"layer{li}.{bi}"
                # residual source
                if blk.downsample is None:
                    res, res_stride = cur, 1
                elif blk.shortcut_type == "A":
                    res, res_stride = cur, s      # strided read, channels < inplanes only (med3d.py:103-112)
                else:  # type B: 1x1x1 strided conv + BN (med3d.py:251-257)
                    wbd = self._conv_bn(name + ".downsample", blk.downsample[0], blk.downsample[1])
                    res = self._add_conv(name + ".downsample", cur, wbd, kernel=1, stride=s, relu=False).out
                    res_stride = 1
                if m.block_kind == "basic":
                    t = self._add_conv(name + ".conv1", cur, self._conv_bn(name + ".conv1", blk.conv1, blk.bn1),
                                       stride=s, dilation=dil).out
                    cur = self._add_conv(name + ".conv2", t, self._conv_bn(name + ".conv2", blk.conv2, blk.bn2),
                                         dilation=dil, residual=res, res_stride=res_stride).out
                else:
                    t = self._add_conv(name + ".conv1", cur, self._conv_bn(name + ".conv1", blk.conv1, blk.bn1),
                                       kernel=1).out
                    t = self._add_conv(name + ".conv2", t, self._conv_bn(name + ".conv2", blk.conv2, blk.bn2),
                                       stride=s, dilation=dil).out
                    cur = self._add_conv(name + ".conv3", t, self._conv_bn(name + ".conv3", blk.conv3, blk.bn3),
                                         kernel=1, residual=res, res_stride=res_stride).out
                inplanes = planes * e
            feats.append(cur)
        x1, x4 = feats[0], feats[3]
        # ---- decoder.  Default: K4 up-samples each stage's input (med3d.py:83, 86) and the first convolution
        # reads it next to the skip tensor.  DRAM_B200_UPSAMPLE=fused moves the up-sampling into that
        # convolution (plane-ring kernel, UP variant; bit-identical results, the up-sampled tensors are never
        # written) — measured slower on B200 (5.9 -> 7.4 ms per 256^3 volume): the interpolation of a chunk's
        # planes cannot overlap the previous chunk's MMAs with only six plane slots, see DESIGN.md.
        fused_up = os.environ.get("DRAM_B200_UPSAMPLE", "separate").lower() == "fused"
        # K4 itself: tensor-core kernel (generated interpolation matrix x source patch) unless DRAM_B200_K4=cuda
        k4_umma = os.environ.get("DRAM_B200_K4", "umma").lower() != "cuda"

        def add_upsample(name, src, dst):
            if k4_umma and src.shape[4] % 64 == 0:
                plan = ops.Upsample2xPlan(src, out=dst)
                self.steps.append(_Step(name, plan.run))
                return plan
            self.steps.append(_Step(name, lambda: ops.upsample2x(src, out=dst)))
            return None

        cb = m.us1.conv_blocks
        # us1.0 (Cin = 512e + 64 -> 64): by default commuted (K13) — 27 channel-mixing products of x4 at LOW
        # resolution, a separable gather, and a 64 -> 64 convolution of the skip tensor that takes the gathered
        # tensor as its residual; DRAM_B200_US1=direct keeps K4 + one convolution over [up(x4) | x1].
        commute = os.environ.get("DRAM_B200_US1", "commute").lower() != "direct"
        if fused_up:
            t = self._add_conv("us1.0", x4, self._conv_bn("us1.0", cb[0][0], cb[0][1]), x2=x1, upsample_x1=True).out
        elif commute:
            t = self._build_commuted_us1(cb[0][0], cb[0][1], x4, x1, (D2, H2, W2), (D3, H3, W3))
        else:
            self.up1 = torch.empty((B, D2, H2, W2, x4.shape[4]), dtype=bf, device=dev)
            add_upsample("us1.upsample", x4, self.up1)
            t = self._add_conv("us1.0", self.up1, self._conv_bn("us1.0", cb[0][0], cb[0][1]), x2=x1).out
        xup1 = self._add_conv("us1.1", t, self._conv_bn("us1.1", cb[1][0], cb[1][1])).out
        cb = m.us2.conv_blocks
        # the full-resolution stage and how far (in voxels) beyond the dRAM's support each step's output is read
        decoder = []
        if fused_up:
            us20 = self._add_conv("us2.0", xup1, self._conv_bn("us2.0", cb[0][0], cb[0][1]), x2=x, upsample_x1=True)
        else:
            self.up2 = torch.empty((B, D1, H1, W1, 64), dtype=bf, device=dev)
            decoder.append(("us2.upsample", add_upsample("us2.upsample", xup1, self.up2), 3, self.up2))
            us20 = self._add_conv("us2.0", self.up2, self._conv_bn("us2.0", cb[0][0], cb[0][1]), x2=x)
        us21 = self._add_conv("us2.1", us20.out, self._conv_bn("us2.1", cb[1][0], cb[1][1]))
        decoder += [("us2.0", us20, 2, us20.out), ("us2.1", us21, 1, us21.out)]
        t, xup2 = us20.out, us21.out
        # ---- us3 + heads fused
        head_ch = tuple(fc.weight.shape[0] for fc in m.fcs)

        def pack_heads():
            w = torch.cat([fc.weight.detach().reshape(fc.weight.shape[0], 32) for fc in m.fcs]).float()
            b = torch.cat([fc.bias.detach() for fc in m.fcs]).float()
            return w.to(dev), b.to(dev)

        hw, hb = pack_heads()
        self._head_w, self._head_b = hw.contiguous(), hb.contiguous()

        def refill_heads():
            w, b = pack_heads()
            self._head_w.copy_(w)
            self._head_b.copy_(b)

        self._packers.append(refill_heads)
        us3 = self._add_conv("us3+heads", xup2, self._conv_bn("us3", m.us3[0], m.us3[1]),
                             heads=(self._head_w, self._head_b, head_ch, self.head_kind == "reg"),
                             store_out=False)
        self.conv_flops += 2 * B * D1 * H1 * W1 * 32 * sum(head_ch)
        self.dense = us3.head_outs
        decoder.append(("us3+heads", us3, 0, None))
        self._decoder = decoder
        # A restricted run writes only around the dRAM's support; the other voxels of these buffers are read (as halo of
        # active items, and by K7's weight-0 corners) but never reach a result: zeros until a run overwrites them.
        for _, _, _, buf in decoder:
            if buf is not None:
                buf.zero_()
        for buf in self.dense:
            buf.zero_()
        self.half_dims = (D1, H1, W1)
        self._plans_alive = [s.fn for s in self.steps]

    def _build_commuted_us1(self, conv, bn, x4, x1, hi, lo):
        """K13 (csrc/upconv_kernels.cu): relu(bn(conv([up(x4) | x1]))) =
        relu(scale * conv(x1, W_skip) + shift + G),  G = sum_tap up(z_tap)[o + tap],  z_tap = (scale * W_up,tap) . x4."""
        dev, bf, B = self.device, self.act_dtype, self.batch
        c_up = x4.shape[4]
        (D2, H2, W2), (D3, H3, W3) = hi, lo

        def pack_z():
            scale, _ = ops.fold_bn(bn, conv.bias)
            packed, mult = ops.pack_upconv_weight(conv.weight.detach().to(dev), c_up, scale.to(dev), dtype=bf)
            return packed, torch.zeros(packed.shape[0], dtype=torch.float32, device=dev), mult

        def pack_skip():
            scale, shift = ops.fold_bn(bn, conv.bias)
            packed, mult = ops.pack_conv_weight(conv.weight.detach().to(dev)[:, c_up:], scale.to(dev), dtype=bf,
                                                normalize=True)
            return packed, shift.to(dev).float(), mult

        m_hi = B * D2 * H2 * W2
        wz = self._register_weight("us1.0.z", pack_z)
        # algorithmic FLOPs: the reference convolves 27 taps of c_up channels at HIGH resolution
        # N tile 256 (an N = 128 tile pulls 128 B/clk/SM of operands through L2 for this short K loop; N = 64 measured
        # 404 TFLOP/s).  Epilogue: staged through shared memory + TMA stores by default — the direct epilogue writes
        # the 3.5 KB rows of z 16 bytes per lane, half a sector each; DRAM_B200_US1_EPILOGUE=direct for A/B runs.
        z_epi = os.environ.get("DRAM_B200_US1_EPILOGUE", "staged").lower()
        z = self._add_conv("us1.0.z", x4, wz, kernel=1, relu=False, flops=2 * m_hi * 64 * c_up * 27, epilogue=z_epi).out
        self.us1_r = torch.empty((B, D3, H3, W2, 9 * 64), dtype=bf, device=dev)
        self.us1_q = torch.empty((B, D3, H2, W2, 3 * 64), dtype=bf, device=dev)
        self.us1_g = torch.empty((B, D2, H2, W2, 64), dtype=bf, device=dev)
        self.steps.append(_Step("us1.0.gather_w", lambda: ops.upconv_axis(z, 3, 9, out=self.us1_r), conv_part=True))
        self.steps.append(_Step("us1.0.gather_h", lambda: ops.upconv_axis(self.us1_r, 2, 3, out=self.us1_q), conv_part=True))
        self.steps.append(_Step("us1.0.gather_d", lambda: ops.upconv_axis(self.us1_q, 1, 1, out=self.us1_g), conv_part=True))
        wskip = self._register_weight("us1.0.skip", pack_skip)
        return self._add_conv("us1.0", x1, wskip, residual=self.us1_g).out

    # ---------------------------------------------------------------- run
    def _launch_steps(self, first=None):
        (first or self.steps[0].fn)()
        self._launch_tail()

    def _launch_tail(self):
        for st in self.steps[1:]:
            st.fn()

    def hu_stem(self, hu, lut, lo=-1150):
        """A replacement for the first recorded step (the stem convolution on `self.image`): the same kernel fed from
        the int16 HU volumes [B,D,H,W] and their window tables (`ops.window_lut`), K8's apply pass folded into a
        gather in its producers.  Pass it to `run_network(first=...)`."""
        if not hasattr(self, "stem_weights"):
            raise RuntimeError("the int16-HU stem needs the fused stem kernel (DRAM_B200_STEM=unfold is set)")
        if tuple(hu.shape) != (self.batch,) + self.dims:
            raise ValueError(f"hu shape {tuple(hu.shape)} does not match the engine's {(self.batch,) + self.dims}")
        w, b, m = self.stem_weights
        return lambda: ops.stem_conv7_hu(hu, lut, w, b, m, out=self.stem_out, lo=lo)

    def image_stem(self, image):
        """A replacement for the first recorded step that reads the caller's fp32 image [B,(1,)D,H,W] in place instead
        of the engine's own input buffer: saves the device-to-device copy of `load_image` (2 x 67 MB per 256^3 volume)
        in `predict_step`.  Pass it to `run_network(first=...)`."""
        if not hasattr(self, "stem_weights"):
            raise RuntimeError("image_stem needs the fused stem kernel (DRAM_B200_STEM=unfold is set)")
        img = image.reshape(self.batch, *self.dims)
        if img.dtype != torch.float32 or not img.is_contiguous():
            raise ValueError("image_stem: expected a contiguous fp32 image")
        w, b, m = self.stem_weights
        return lambda: ops.stem_conv7(img, w, b, m, out=self.stem_out)

    def _restricted_tail(self):
        """Launches of the recorded sequence after the first step, with the full-resolution decoder steps restricted to
        the work items the dRAM of the ess mask reaches (needs `self._restricted` filled by `_support`)."""
        for fn in self._restricted[2]:
            fn()

    def _support(self, ess):
        """Eager part of a restricted run: the support bits of `ess` uint8 [B, D, H, W] on the decoder grid."""
        if tuple(ess.shape) != (self.batch,) + self.dims or ess.dtype != torch.uint8 or not ess.is_contiguous():
            raise ValueError(f"active_ess: expected contiguous uint8 {(self.batch,) + self.dims}, got "
                             f"{ess.dtype} {tuple(ess.shape)}")
        if self._restricted is None:
            B, (D, H, W), (d, h, w) = self.batch, self.dims, self.half_dims
            words = (w + 31) // 32
            rows = torch.empty((B, D, H, words), dtype=torch.int32, device=self.device)
            support = torch.empty((B, d, h, words), dtype=torch.int32, device=self.device)
            lists, listed = [], {}
            for name, plan, radius, _ in self._decoder:
                size = plan.worklist_size() if plan is not None else 0
                if size == 0:
                    continue   # a kernel without work lists (selected by a DRAM_B200_* experiment switch) stays dense
                flags = torch.empty(size, dtype=torch.uint8, device=self.device)
                items = torch.empty(size, dtype=torch.int32, device=self.device)
                count = torch.empty(1, dtype=torch.int32, device=self.device)
                lists.append(lambda plan=plan, r=radius, f=flags, i=items, c=count: plan.build_worklist(support, r, f, i, c))
                listed[name] = lambda plan=plan, i=items, c=count: plan.run_listed(i, c)
            self._restricted = (rows, support, lists + [listed.get(st.name, st.fn) for st in self.steps[1:]])
        rows, support, _ = self._restricted
        ops.decoder_support(ess, self.half_dims, rows=rows, out=support)

    def run_network(self, first=None, active_ess=None):
        """The recorded launch sequence on `self.image` -> `self.dense` (engine-owned), on the current stream.
        `first` replaces the first step (see `hu_stem`); it is launched eagerly, the rest replays as a graph.
        `active_ess` (uint8 [B, D, H, W], the ess mask K7 will apply): the dense maps are computed only where K7 reads
        them for this mask — the full-resolution decoder steps run the work items that reach those voxels, with the same
        arithmetic, so the dRAM is bit-identical to a dense run's; elsewhere the maps hold stale finite values.  The
        mask is read by an eager launch in front of the graph (its address changes from call to call).

        * fp16 storage: the first pass after the weights changed (`DRAM_B200_SAT_CHECK=first`, default; `always` /
          `off`) runs with the library's saturation probe on and raises `ops.ActivationOverflow` if any convolution
          output left the fp16 range (the epilogue clamps to +-65504 silently otherwise) — one 4-byte read-back.
        * afterwards the sequence is one CUDA graph (captured on first use, `DRAM_B200_GRAPH=0` keeps eager
          launches): every buffer the kernels touch is engine-owned and address-stable, so a replay is exact."""
        if self._weights_epoch != self.model.weights_epoch:
            self.refresh_weights()
        mode = ops.sat_check_mode()
        if self.act_dtype == torch.float16 and (
                mode == "always" or (mode == "first" and self._sat_checked_epoch != self._weights_epoch)):
            lib = ops._capi.load()
            self._sat_counter.zero_()
            ops.check(lib.dram_set_saturation_counter(ops._p(self._sat_counter)), "dram_set_saturation_counter")
            try:
                self._launch_steps(first)   # dense, also for a restricted call: the probe covers every voxel
            finally:
                lib.dram_set_saturation_counter(None)
            clamped = int(self._sat_counter.item())
            self.last_saturation_count = clamped
            if clamped:
                raise ops.ActivationOverflow(
                    f"{clamped} 32-channel output groups exceeded the fp16 range (+-65504) and were clamped: this "
                    "checkpoint/input needs bf16 storage (model.act_dtype = torch.bfloat16 or DRAM_B200_DTYPE=bf16)")
            self._sat_checked_epoch = self._weights_epoch
            return self.dense
        tail = self._launch_tail
        if active_ess is not None:
            self._support(active_ess)
            tail = self._restricted_tail
        if not ops.graphs_enabled() or torch.cuda.is_current_stream_capturing():
            (first or self.steps[0].fn)()
            tail()
            return self.dense
        (first or self.steps[0].fn)()   # the stem reads a caller-owned buffer in the HU variant: outside the graph
        attr = "_graph" if active_ess is None else "_graph_restricted"
        if getattr(self, attr) is None:
            tail()  # warm-up outside the capture (lazy function attributes, module loading)
            torch.cuda.current_stream(self.device).synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                tail()
            setattr(self, attr, graph)
        getattr(self, attr).replay()
        return self.dense

    def load_image(self, image):
        """Copies fp32 [B,(1,)D,H,W] into the engine's input buffer (no-op when it already is that buffer)."""
        img = image.reshape(self.batch, *self.dims)
        if img.data_ptr() != self.image.data_ptr():
            self.image.copy_(img)

    def run(self, image, lungs=None):
        """image: fp32 [B, D, H, W] (or [B,1,D,H,W]) on the device.  lungs: None, uint8/bool [B,D,H,W]
        or float [B,(1,)D,H,W].  Returns (dense list fp32 [B,C,d,h,w] — engine-owned buffers that the
        next run overwrites — and the pooled scores list)."""
        B = self.batch
        self.load_image(image)
        self.run_network()
        mask = None
        if lungs is not None:
            mask = lungs.reshape(B, *lungs.shape[-3:])
            if mask.dtype == torch.bool:
                mask = mask.view(torch.uint8)
            elif mask.dtype != torch.uint8:
                mask = mask.to(torch.float32)
            mask = mask.contiguous()
        pooled = [ops.masked_pool(d, mask if self.head_kind == "reg" else None) for d in self.dense]
        if self.head_kind == "reg":
            pooled = [p.reshape(B) for p in pooled]
        return self.dense, pooled

    def launches_per_run(self):
        """Kernel launches of one run(): recorded steps + 2 pooling calls x (partial + finalize)."""
        return len(self.steps) + 4
