"""The full-resolution decoder restricted to the dRAM's support (`run_network(active_ess=...)`, used by predict_step and
predict_step_from_hu): the support bits and the work lists against numpy, guard bands of the builder's writes, and
every returned tensor bit-identical to the dense route (run_network() then K7) over ess masks that cross item and volume
borders, for all three *dram architectures, ragged shapes, eager launches and graph replays with a new mask per call."""
from argparse import Namespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import pipeline_oracle as P
from oracle import synthetic

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ numpy reference
def _corners(n_out, n_in):
    """K7's source indices (i0, i1) per output index: ATen's align_corners rule in fp32 (lin_index_ac)."""
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0)
    i0 = np.minimum((np.float32(scale) * np.arange(n_out, dtype=np.float32)).astype(np.int64), n_in - 1)
    return i0, i0 + (i0 < n_in - 1)


def ref_support(ess, half):
    """R0: the decoder-grid voxels K7 reads for ess [B, D, H, W] -> bool [B, d, h, w]."""
    B, D, H, W = ess.shape
    idx = [_corners(n, m) for n, m in zip((D, H, W), half)]
    out = np.zeros((B,) + tuple(half), dtype=bool)
    b, z, y, x = np.nonzero(ess)
    for cz in idx[0]:
        for cy in idx[1]:
            for cx in idx[2]:
                out[b, cz[z], cy[y], cx[x]] = True
    return out


def ref_items(support, radius, tile, d_fastest):
    """Ascending indices of the tiles (tw, th, td) whose box grown by `radius` meets `support`."""
    m = torch.from_numpy(support)[:, None].float()
    if radius:
        m = F.max_pool3d(m, 2 * radius + 1, 1, radius)
    tw, th, td = tile
    B, _, d, h, w = m.shape
    m = F.pad(m, (0, -w % tw, 0, -h % th, 0, -d % td))
    act = F.max_pool3d(m, (td, th, tw), (td, th, tw))[:, 0] > 0          # [B, tiles_d, tiles_h, tiles_w]
    if d_fastest:
        act = act.permute(0, 2, 3, 1)
    return np.nonzero(act.reshape(-1).numpy())[0]


def _unpack(bits, w):
    b = bits.cpu().numpy().view(np.uint8)
    full = np.unpackbits(b, axis=-1, bitorder="little")
    return full[..., :w].astype(bool), full[..., w:]


def _ess_cases(B, dims, seed):
    D, H, W = dims
    g = torch.Generator().manual_seed(seed)
    cases = {"zero": torch.zeros((B, D, H, W), dtype=torch.uint8), "one": torch.ones((B, D, H, W), dtype=torch.uint8)}
    c = torch.zeros((B, D, H, W), dtype=torch.uint8)
    for z in (0, D - 1):
        for y in (0, H - 1):
            for x in (0, W - 1):
                c[:, z, y, x] = 1
    cases["corners"] = c
    # single voxels on the faces of 8 x 16 x 4 items of the decoder grid (full-grid voxels 2x, 2x +- 1 of those faces)
    f = torch.zeros((B, D, H, W), dtype=torch.uint8)
    for b in range(B):
        for k in range(6):
            z = min(2 * (4 * (k + 1)) - 1 + (b + k) % 3, D - 1)
            y = min(2 * 16 - 1 + k % 2, H - 1)
            x = min(2 * 8 * (k % 3 + 1) - (k + b) % 3, W - 1)
            f[b, z, y, x] = 1
    cases["faces"] = f
    cases["sparse"] = (torch.rand((B, D, H, W), generator=g) < 2e-4).to(torch.uint8)
    vols = [synthetic.make_volume(70 + seed + b, dims) for b in range(B)]
    cases["volumes"] = torch.stack([((v[0] < -910) & (v[1] > 0)).to(torch.uint8) for v in vols])
    return cases, torch.stack([v[0] for v in vols]), torch.stack([(v[1] > 0).to(torch.uint8) for v in vols])


# ------------------------------------------------------------------------------------------------ builder
@pytest.mark.parametrize("shape", [(2, 64, 64, 64), (1, 63, 71, 40), (3, 31, 32, 47)])
def test_support_and_worklists_match_numpy(cuda, lib, shape):
    from dram_b200 import ops

    B, D, H, W = shape
    half = tuple((n - 1) // 2 + 1 for n in (D, H, W))
    cases, _, _ = _ess_cases(B, (D, H, W), seed=1)
    x = torch.zeros((B,) + half + (64,), dtype=torch.float16, device=cuda)
    bias = torch.zeros(64, dtype=torch.float32, device=cuda)
    w64 = torch.zeros((64, 27 * 64), dtype=torch.float16, device=cuda)
    ring = ops.Conv3dPlan(x, w64, bias)                        # 64 -> 64 plane ring: 8 x 16 x 4 items
    stream = ops.Conv3dPlan(x, w64[:32].contiguous(), bias[:32].contiguous())   # 64 -> 32 streaming: plane steps
    lo = torch.zeros((B,) + tuple(n // 2 for n in half) + (64,), dtype=torch.float16, device=cuda)
    plans = [(ring, (8, 16, 4), True), (stream, (8, 16, 1), True)]
    if all(n % 2 == 0 for n in half):
        plans.append((ops.Upsample2xPlan(lo, out=torch.zeros_like(x)), (8, 4, 4), False))
    for name, ess in cases.items():
        want = ref_support(ess.numpy(), half)
        bits = ops.decoder_support(ess.to(cuda), half)
        got, pad = _unpack(bits, half[2])
        assert np.array_equal(got, want), name
        assert not pad.any(), name
        for plan, tile, d_fastest in plans:
            size = plan.worklist_size()
            flags = torch.empty(size, dtype=torch.uint8, device=cuda)
            items = torch.full((size,), -1, dtype=torch.int32, device=cuda)
            count = torch.full((1,), -1, dtype=torch.int32, device=cuda)
            for radius in (0, 1, 2, 3):
                plan.build_worklist(bits, radius, flags, items, count)
                ref = ref_items(want, radius, tile, d_fastest)
                n = int(count.item())
                assert n == len(ref), (name, tile, radius)
                assert np.array_equal(items[:n].cpu().numpy(), ref), (name, tile, radius)


def test_worklist_builder_stays_inside_its_buffers(cuda, lib):
    from dram_b200 import ops

    PAD = 4096

    def guarded(n, dtype):
        item = torch.empty((), dtype=dtype).element_size()
        raw = torch.full((2 * PAD + n * item,), 0xA5, dtype=torch.uint8, device=cuda)
        return raw, raw[PAD:PAD + n * item].view(dtype)

    def untouched(raw, what):
        torch.cuda.synchronize()
        assert bool((raw[:PAD] == 0xA5).all()) and bool((raw[-PAD:] == 0xA5).all()), what

    B, D, H, W = 1, 39, 47, 71
    half = tuple((n - 1) // 2 + 1 for n in (D, H, W))
    words = (half[2] + 31) // 32
    ess = torch.ones((B, D, H, W), dtype=torch.uint8, device=cuda)
    rows_raw, rows = guarded(B * D * H * words, torch.int32)
    bits_raw, bits = guarded(B * half[0] * half[1] * words, torch.int32)
    ops.decoder_support(ess, half, rows=rows.view(B, D, H, words), out=bits.view(B, half[0], half[1], words))
    untouched(rows_raw, "support rows")
    untouched(bits_raw, "support bits")
    x = torch.zeros((B,) + half + (64,), dtype=torch.float16, device=cuda)
    plan = ops.Conv3dPlan(x, torch.zeros((64, 27 * 64), dtype=torch.float16, device=cuda),
                          torch.zeros(64, dtype=torch.float32, device=cuda))
    size = plan.worklist_size()
    (f_raw, flags), (i_raw, items), (c_raw, count) = (guarded(size, torch.uint8), guarded(size, torch.int32),
                                                      guarded(1, torch.int32))
    plan.build_worklist(bits.view(B, half[0], half[1], words), 3, flags, items, count)
    for raw, what in ((f_raw, "flags"), (i_raw, "items"), (c_raw, "count")):
        untouched(raw, what)
    assert int(count.item()) == size


# ------------------------------------------------------------------------------------------------ end to end
def _module(arch, sd, cuda):
    from dram_b200.models import ScanRegLightningModule

    module = ScanRegLightningModule(Namespace(model_arch=arch))
    module.model.load_state_dict(sd)
    return module.to(cuda).eval()


def _dense_route(module, eng, ess, lungs, dims, first=None):
    from dram_b200 import ops

    dense = eng.run_network(first=first)
    cle, pse, pct = ops.dram_upsample_mask(dense[0], dense[1], ess, lungs, dims)
    return {"cle_dense_outs": cle, "pse_dense_outs": pse, "cle_precentages": pct[0], "pse_precentages": pct[1]}


def _assert_equal(got, want, what):
    for k, v in want.items():
        assert torch.equal(got[k], v), f"{what}: {k}"


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("arch,dims,B", [("med3ddram18", (32, 32, 32), 1), ("med3ddram18", (39, 48, 63), 3),
                                         ("med3ddram", (64, 64, 64), 1), ("med3ddram50", (47, 40, 32), 3)])
def test_restricted_decoder_is_bit_identical_to_dense(cuda, lib, monkeypatch, graph, arch, dims, B):
    from dram_b200 import ops

    monkeypatch.setenv("DRAM_B200_GRAPH", graph)
    sd = synthetic.make_state_dict(arch, seed=3, calib_dims=dims)
    module = _module(arch, sd, cuda)
    cases, hu_a, lungs = _ess_cases(B, dims, seed=B)
    hu_a, lungs = hu_a.to(cuda), lungs.to(cuda)
    hu_b = hu_a.flip(1).contiguous()    # another input: its activations are what a restricted run must not pass on
    eng = module.model.engine(B, dims, cuda)
    image = torch.stack([P.standardize(P.intensity_window(h)) for h in hu_a.cpu()]).to(cuda).contiguous()
    runs = []
    # a dense run of the other input before each restricted call: stale activations everywhere outside the support
    for name, ess in cases.items():
        ess = ess.to(cuda)
        ops.window_standardize(hu_b, out=eng.image, batched=True)
        eng.run_network()
        runs.append(("from_hu " + name, hu_a, ess, module.predict_step_from_hu(hu_a, lungs, ess)))
        eng.run_network()
        batch = {"image": image, "lung_mask": lungs.bool(), "ess_mask": ess.bool()}
        runs.append(("predict_step " + name, None, ess, module.predict_step(batch, 0)))
    # restricted calls back to back, inputs alternating, a new mask each time
    for i, name in enumerate(("volumes", "sparse", "faces", "zero", "one", "corners")):
        hu, ess = (hu_a, hu_b)[i % 2], cases[name].to(cuda)
        runs.append(("again " + name, hu, ess, module.predict_step_from_hu(hu, lungs, ess)))
    for what, hu, ess, got in runs:
        if hu is None:
            want = _dense_route(module, eng, ess, lungs, dims, first=eng.image_stem(image))
        else:
            ops.window_standardize(hu, out=eng.image, batched=True)
            want = _dense_route(module, eng, ess, lungs, dims)
        _assert_equal(got, want, what)


def test_restricted_run_uses_the_lists_and_follows_the_support(cuda, lib, monkeypatch):
    """The restricted route really skips work: after a dense run of another input, the maps it leaves hold that input's
    values away from the support and the dense values on it; graph replay and eager launches leave the same buffers."""
    from dram_b200 import ops

    arch, dims, B = "med3ddram18", (32, 48, 64), 2
    module = _module(arch, synthetic.make_state_dict(arch, seed=5, calib_dims=dims), cuda)
    cases, hu_a, lungs = _ess_cases(B, dims, seed=7)
    hu_a, lungs, ess = hu_a.to(cuda), lungs.to(cuda), cases["sparse"].to(cuda)
    hu_b = hu_a.flip(2).contiguous()
    eng = module.model.engine(B, dims, cuda)
    maps, outs = {}, {}
    for graph in ("1", "0"):
        monkeypatch.setenv("DRAM_B200_GRAPH", graph)
        ops.window_standardize(hu_b, out=eng.image, batched=True)
        eng.run_network()
        outs[graph] = module.predict_step_from_hu(hu_a, lungs, ess)
        maps[graph] = [t.clone() for t in eng.dense]
    assert eng._graph_restricted is not None
    _assert_equal(outs["0"], outs["1"], "eager vs graph")
    assert all(torch.equal(a, b) for a, b in zip(maps["0"], maps["1"]))
    ops.window_standardize(hu_a, out=eng.image, batched=True)
    dense = [t.clone() for t in eng.run_network()]
    support = torch.from_numpy(ref_support(ess.cpu().numpy(), eng.half_dims)).to(cuda)[:, None]
    assert 0 < int(support.sum()) < support.numel() // 4
    for got, want in zip(maps["1"], dense):
        assert torch.equal(got[support], want[support])
        assert not torch.equal(got, want), "the restricted run computed the maps everywhere"
