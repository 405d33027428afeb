"""Sample-folded bricks of the tile kernels (conv3d_umma.cu, conv3d_pair.cu).

A brick may span tn samples at the same spatial position, so that its spatial extents line up with a dilated
filter's zero padding and more padding taps are skipped.  Every folded plan is bit-equal (`torch.equal`) to the same
convolution forced to the unfolded 8x4x4 layout (explicit tile = one sample per brick), and within the tolerance of
test_conv3d_gpu.py of torch: |err| <= 2^-7 * |ref| + 2^-8 * max|ref|.  The reference is an fp32 convolution on the
GPU with TF32 off, so the layer3 / layer4 shapes at batch 4 stay quick.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _close(got, ref, what):
    err = (got - ref).abs()
    tol = ref.abs() * 2.0 ** -7 + ref.abs().max() * 2.0 ** -8
    bad = err > tol
    assert not bad.any(), f"{what}: {int(bad.sum())}/{bad.numel()} outside tolerance; max err {err.max().item():.4g}"


def _operands(cuda, n, dims, cin, cout, res_c, dt, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((n, cin) + dims, generator=g).to(dt)
    w = (torch.randn((cout, cin, 3, 3, 3), generator=g) * (27 * cin) ** -0.5).to(dt)
    b = torch.randn(cout, generator=g) * 0.1
    res = torch.randn((n, res_c) + dims, generator=g).to(dt) if res_c else None
    return x.to(cuda), w.to(cuda), b.to(cuda), None if res is None else res.to(cuda)


def _reference(x, w, b, res, dil):
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        ref = F.conv3d(x.float(), w.float(), b, padding=dil, dilation=dil)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    if res is not None:
        ref[:, :res.shape[1]] += res.float()
    return ref.relu()


def _plan(ops, x, w, b, res, dil, dt, tile=None, out=None):
    return ops.Conv3dPlan(ops.to_ndhwc_16(x.float(), dt), ops.pack_conv_weight(w.float(), dtype=dt), b, kernel=3,
                          dilation=dil, residual=None if res is None else ops.to_ndhwc_16(res.float(), dt), tile=tile,
                          out=out)


FOLD_CASES = [
    # (batch, (D, H, W), cin, cout, dilation, res_c, pair knob, max_ctas, expected brick (w, h, d, samples), pair)
    (4, (32, 32, 32), 256, 256, 2, 256, None, 0, (16, 2, 2, 2), False),  # layer3 at batch 4
    (4, (32, 32, 32), 256, 512, 4, 0, None, 0, (4, 4, 4, 2), False),     # layer4.0.conv1 at batch 4
    (4, (32, 32, 32), 512, 512, 4, 512, None, 0, (4, 4, 4, 4), True),    # layer4 at batch 4: pair kernel
    (4, (32, 32, 32), 512, 512, 4, 0, "0", 3, (4, 4, 4, 2), False),      # layer4, pair kernel off, 3 CTAs
    (3, (8, 8, 8), 256, 256, 4, 256, "0", 0, (4, 4, 4, 2), False),       # ragged batch: tn = 2, sample 3 is past n
    (3, (8, 8, 8), 256, 256, 2, 0, "0", 1, (8, 2, 2, 4), False),         # ragged batch: tn = 4, one CTA
    (3, (8, 8, 8), 256, 512, 4, 512, "1", 3, (4, 4, 4, 4), True),        # pair: second box holds samples 2, 3
    (3, (4, 8, 8), 256, 256, 2, 0, "1", 1, (8, 8, 2, 2), True),          # pair: one sample per box, sample 3 past n
    (3, (6, 10, 10), 256, 256, 4, 256, "0", 3, (4, 4, 2, 4), False),     # ragged spatial sizes and batch
    (3, (6, 10, 10), 256, 256, 4, 0, "1", 1, (16, 2, 2, 4), True),
    (2, (5, 9, 7), 128, 256, 2, 128, "0", 0, (8, 4, 2, 2), False),       # shortcut-A residual (res_c < cout)
]


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("case", range(len(FOLD_CASES)))
def test_folded_plan_matches_unfolded(cuda, lib, case, dt, monkeypatch):
    from dram_b200 import ops

    n, dims, cin, cout, dil, res_c, knob, max_ctas, brick, pair = FOLD_CASES[case]
    if knob is None:
        monkeypatch.delenv("DRAM_B200_PAIR_TILES", raising=False)
    else:
        monkeypatch.setenv("DRAM_B200_PAIR_TILES", knob)
    x, w, b, res = _operands(cuda, n, dims, cin, cout, res_c, dt, seed=300 + case)
    folded = _plan(ops, x, w, b, res, dil, dt)
    assert folded.brick == brick and folded.pair == pair, (folded.brick, folded.pair)
    got = folded.run(max_ctas).clone()
    unfolded = _plan(ops, x, w, b, res, dil, dt, tile=(8, 4, 4))
    assert unfolded.brick == (8, 4, 4, 1) and not unfolded.pair
    assert folded.executed_flops < unfolded.executed_flops
    want = unfolded.run().clone()
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    _close(ops.to_ncdhw_f32(got), _reference(x, w, b, res, dil), f"folded {brick} pair={pair} {dims} n={n} {dt}")


@pytest.mark.parametrize("knob", ["0", "1"])
def test_folded_ragged_batch_guard_band(cuda, lib, knob, monkeypatch):
    """The rows of samples past the batch are never stored: the output is a view between two sentinel samples."""
    from dram_b200 import ops

    monkeypatch.setenv("DRAM_B200_PAIR_TILES", knob)
    n, dims, dil, dt = 3, (8, 8, 8), 4, torch.bfloat16
    x, w, b, res = _operands(cuda, n, dims, 256, 256, 256, dt, seed=77)
    big = torch.full((n + 2,) + dims + (256,), -77.5, dtype=dt, device=cuda)
    before = big.clone()
    plan = _plan(ops, x, w, b, res, dil, dt, out=big[1:n + 1])
    assert plan.brick[3] in (2, 4) and plan.pair == (knob == "1"), plan.brick  # the last group holds sample 3
    plan.run(2)
    torch.cuda.synchronize()
    assert torch.equal(big[0], before[0]) and torch.equal(big[n + 1], before[n + 1])
    want = _plan(ops, x, w, b, res, dil, dt, tile=(8, 4, 4)).run()
    torch.cuda.synchronize()
    assert torch.equal(big[1:n + 1], want)


def _axis_taps(out, ext, dil):
    """Taps a row of bricks of `ext` outputs executes along one axis (stride 1, padding = dilation)."""
    return sum(1 for b0 in range(0, out, ext) for z in range(3)
               if not (b0 + z * dil - dil + ext - 1 < 0 or b0 + z * dil - dil >= out))


def _model_stages(n, size, dil, brick):
    bw, bh, bd, bn = brick
    groups = -(-n // bn)
    return groups * _axis_taps(size, bw, dil) * _axis_taps(size, bh, dil) * _axis_taps(size, bd, dil)


@pytest.mark.parametrize("batch", [1, 4])
def test_executed_flops_stage_model(cuda, lib, batch, monkeypatch):
    """executed_flops counts the (brick, tap) stages of the chosen brick: layer3 and layer4 of the default network
    (32^3 maps) fold at batch 4 (8.2 % / 8.3 % fewer stages than 8x4x4 bricks) and are unchanged at batch 1."""
    from dram_b200 import ops

    monkeypatch.delenv("DRAM_B200_PAIR_TILES", raising=False)
    dt = torch.bfloat16
    size = 32
    expect = {4: {"layer3": ((16, 2, 2, 2), False, 25392, 27648), "layer4": ((4, 4, 4, 4), True, 2 * 10648, 23232)},
              1: {"layer3": ((8, 4, 4, 1), False, 6912, 6912), "layer4": ((8, 4, 4, 1), False, 5808, 5808)}}[batch]
    for name, cin, dil in (("layer3", 256, 2), ("layer4", 512, 4)):
        x = torch.zeros((batch, size, size, size, cin), dtype=dt, device=cuda)
        w = torch.zeros((cin, 27 * cin), dtype=dt, device=cuda)
        b = torch.zeros(cin, device=cuda)
        plan = ops.Conv3dPlan(x, w, b, kernel=3, dilation=dil)
        old = ops.Conv3dPlan(x, w, b, kernel=3, dilation=dil, tile=(8, 4, 4))
        brick, pair, stages, old_stages = expect[name]
        assert plan.brick == brick and plan.pair == pair, (name, plan.brick, plan.pair)
        boxes = 2 if plan.pair else 1
        assert _model_stages(batch, size, dil, brick) * boxes == stages
        assert _model_stages(batch, size, dil, (8, 4, 4, 1)) == old_stages
        per_stage = 2 * 128 * plan.block_n * plan.n_tiles * (cin // 64) * 64
        assert plan.executed_flops == stages * per_stage, name
        assert old.executed_flops == old_stages * 2 * 128 * old.block_n * old.n_tiles * (cin // 64) * 64, name


def _host_tile_order(plan, dims, dil):
    """The stable descending-cost permutation of the plan's tiles, from the brick geometry (n-tile fastest)."""
    bw, bh, bd, bn = plan.brick
    n = plan.out_shape[0]
    size_d, size_h, size_w = dims

    def taps(out, ext):
        return [sum(1 for z in range(3) if not (b0 + z * dil - dil + ext - 1 < 0 or b0 + z * dil - dil >= out))
                for b0 in range(0, out, ext)]

    tw, th, td = taps(size_w, bw), taps(size_h, bh), taps(size_d, bd)
    cost = [td[d] * th[h] * tw[w] for _ in range(-(-n // bn)) for d in range(len(td)) for h in range(len(th))
            for w in range(len(tw))]
    ms = sorted(range(len(cost)), key=lambda m: -cost[m])   # sorted() is stable
    return [m * plan.n_tiles + t for m in ms for t in range(plan.n_tiles)]


@pytest.mark.parametrize("n,dims,cin,cout,dil,knob", [
    (4, (32, 32, 32), 512, 512, 4, None),   # layer4 pair plan at batch 4
    (1, (32, 32, 32), 512, 512, 4, None),   # layer4 at batch 1: unfolded 8x4x4, border bricks still cheaper
    (3, (6, 10, 10), 256, 256, 4, "0"),     # ragged, folded
])
def test_tile_order_built_on_device(cuda, lib, n, dims, cin, cout, dil, knob, monkeypatch):
    """The order the device builds into the plan's caller-owned buffer is the stable descending-cost permutation."""
    from dram_b200 import ops

    if knob is None:
        monkeypatch.delenv("DRAM_B200_PAIR_TILES", raising=False)
    else:
        monkeypatch.setenv("DRAM_B200_PAIR_TILES", knob)
    x = torch.zeros((n,) + dims + (cin,), dtype=torch.bfloat16, device=cuda)
    plan = ops.Conv3dPlan(x, torch.zeros((cout, 27 * cin), dtype=torch.bfloat16, device=cuda),
                          torch.zeros(cout, device=cuda), kernel=3, dilation=dil)
    assert plan.tile_order is not None
    assert plan.tile_order.cpu().tolist() == _host_tile_order(plan, dims, dil)
    # dilation 1: every brick executes every tap, no order
    plan1 = ops.Conv3dPlan(x, torch.zeros((cout, 27 * cin), dtype=torch.bfloat16, device=cuda),
                           torch.zeros(cout, device=cuda), kernel=3, dilation=1, algo="tiles")
    assert plan1.tile_order is None


@pytest.mark.parametrize("n,cin", [(2, 256), (1, 64)])
def test_dilated_conv_op_captures_in_a_graph(cuda, lib, n, cin):
    """dram_b200::conv3d with dilation 4 builds its plan (tensor maps, tile order) inside a CUDA graph capture: no
    allocation outside the caching allocator, no synchronisation; the replay follows new input data."""
    from dram_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(5)
    dt = torch.float16
    xs = torch.randn((n, 8, 12, 16, cin), generator=g, device=cuda).to(dt)
    w = torch.randn((cin, cin, 3, 3, 3), generator=g, device=cuda) * (27 * cin) ** -0.5
    packed, bias = ops.pack_conv_weight(w, dtype=dt), torch.zeros(cin, device=cuda)
    probe = ops.Conv3dPlan(xs, packed, bias, kernel=3, dilation=4)
    assert probe.tile_order is not None
    torch.ops.dram_b200.conv3d(xs, packed, bias, dilation=4)  # warm-up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = torch.ops.dram_b200.conv3d(xs, packed, bias, dilation=4)
    for _ in range(2):
        xs.copy_(torch.randn(xs.shape, generator=g, device=cuda).to(dt))
        graph.replay()
        torch.cuda.synchronize()
        want = ops.Conv3dPlan(xs, packed, bias, kernel=3, dilation=4).run()
        torch.cuda.synchronize()
        assert torch.equal(out, want)
