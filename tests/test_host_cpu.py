"""CPU-only checks of the host side: the C-ABI library loads and exports every declared symbol, argument
validation works without a GPU, and the drop-in Python surface (factories, state_dict layout, config
resolution, checkpoint loading, sharding, .mha I/O, labels, result merging) behaves like the reference's."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol(lib):
    from dram_b200 import _capi

    header = open(os.path.join(ROOT, "include", "dram_b200.h")).read()
    declared = set(re.findall(r"\b(dram_[a-z0-9_]+)\s*\(", header))
    declared -= {"dram_last_error"} - {"dram_last_error"}
    assert declared, "no declarations parsed"
    assert declared == set(_capi.SIGNATURES), (declared ^ set(_capi.SIGNATURES))
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in include/dram_b200.h but not exported"
    assert lib.dram_version() == 5


def test_argument_validation_without_gpu(lib):
    import ctypes as C

    from dram_b200 import _capi

    d = _capi.ConvDesc()
    handle = C.c_void_p()
    rc = lib.dram_conv3d_plan_create(C.byref(d), None, None, None, None, None, None, None, None, None, None, None,
                                     C.byref(handle))
    assert rc == -1 and "required" in _capi.last_error()
    d.n, d.di, d.hi, d.wi, d.c1, d.cout = 1, 8, 8, 8, 60, 64
    d.kd = d.kh = d.kw = 3
    d.sd = d.sh = d.sw = d.dd = d.dh = d.dw = 1
    rc = lib.dram_conv3d_plan_create(C.byref(d), 16, None, 16, 16, None, None, 16, None, None, None, None, C.byref(handle))
    assert rc == -1 and "multiple of 64" in _capi.last_error()
    do, ho, wo = C.c_int32(), C.c_int32(), C.c_int32()
    d.di, d.hi, d.wi, d.pd, d.ph, d.pw, d.sd = 256, 128, 128, 3, 0, 0, 2
    d.kd, d.kh, d.kw = 7, 1, 1
    assert lib.dram_conv3d_out_dims(C.byref(d), C.byref(do), C.byref(ho), C.byref(wo)) == 0
    assert (do.value, ho.value, wo.value) == (128, 128, 128)
    assert lib.dram_maxpool3d(None, None, 1, 8, 8, 8, 64, 0, None) == -1
    assert lib.dram_stem_expand(None, None, 1, 8, 8, 8, 7, None) == -1  # bad dtype code
    assert lib.dram_pool_workspace_bytes(2, 3) == 8 * 2 * 4
    # K11 / K12 (training tail): null pointers, batch bound, step count from 1, alignment
    assert lib.dram_train_loss_workspace_bytes(2) >= 2 * 8 * 8
    assert lib.dram_train_loss_forward(*([None] * 10), 2, 8, 8, 8, 4, 4, 4, 0.7, 0.25, None, None, None) == -1
    assert "null pointer" in _capi.last_error()
    assert lib.dram_train_loss_forward(*([16] * 10), 65, 8, 8, 8, 4, 4, 4, 0.7, 0.25, 16, 16, None) == -1
    assert "batch 65" in _capi.last_error()
    assert lib.dram_train_loss_backward(*([16] * 7), None, 1, 8, 8, 8, 4, 4, 0, 16, 16, None) == -1
    assert lib.dram_peer_exchange_bytes() >= 4 * 8 * 4096 * 8
    assert lib.dram_peer_allreduce_f64(None, None, 8, None, 2, 0, 1, None, None) == -1
    assert lib.dram_peer_open(None, None) == -1 and lib.dram_peer_close(None) == -1 and lib.dram_peer_free(None) == -1
    assert lib.dram_adam_step(None, None, None, None, 8, 1e-4, 0.9, 0.999, 1e-8, 1, 1.0, None) == -1
    assert lib.dram_adam_step(16, 16, 16, 16, 8, 1e-4, 0.9, 0.999, 1e-8, 0, 1.0, None) == -1
    assert "counts from 1" in _capi.last_error()
    assert lib.dram_adam_step(16, 16, 20, 16, 8, 1e-4, 0.9, 0.999, 1e-8, 1, 1.0, None) == -1
    assert "aligned" in _capi.last_error()


def test_ops_refuse_cpu_tensors(lib):
    from dram_b200 import ops

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.maxpool3d(torch.zeros(1, 4, 4, 4, 64, dtype=torch.bfloat16))
    with pytest.raises(RuntimeError):
        ops.window_standardize(torch.zeros(4, 4, 4, dtype=torch.int16))


def test_factories_and_state_dict_layout():
    from dram_b200 import med3d

    with open(os.path.join(GOLDEN, "state_layouts.json")) as f:
        layouts = json.load(f)
    fac = {"med3d": med3d.resnet34segcls, "med3d18": med3d.resnet18segcls, "med3d50": med3d.resnet50segcls,
           "med3ddram": med3d.resnet34segreg, "med3ddram18": med3d.resnet18segreg, "med3ddram50": med3d.resnet50segreg}
    for arch, f in fac.items():
        m = f(n_classes=[6, 3]) if "dram" not in arch else f()
        got = [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()]
        assert got == layouts[arch]["keys"], arch
        assert type(m).__name__ == layouts[arch]["class"]
        assert m.get_target_layer() is m.us3
        assert sum(p.numel() for p in m.parameters()) == layouts[arch]["params"]


def test_get_model_by_name_and_greedy_load(tmp_path):
    from dram_b200 import utils

    m = utils.get_model_by_name("med3ddram18")
    assert type(m).__name__ == "ResNetSegReg" and len(m.state_dict()) == 141
    c = utils.get_model_by_name("med3d18")
    assert type(c).__name__ == "ResNetSegCls" and c.n_classes == [6, 3]
    with pytest.raises(FileNotFoundError):
        utils.get_model_by_name("nope")
    sd = {k: torch.full_like(v, 0.5) if v.is_floating_point() else v for k, v in m.state_dict().items()}
    sd["conv1.weight"] = torch.zeros(3, 3)      # shape mismatch -> skipped
    sd["not.a.key"] = torch.zeros(1)            # unexpected -> skipped
    del sd["bn1.bias"]                          # missing -> kept
    before = m.conv1.weight.clone()
    utils.load_state_dict_greedy(m, sd)
    assert torch.equal(m.conv1.weight, before)
    assert float(m.layer1[0].conv1.weight.mean()) == 0.5
    # Lightning checkpoints carry the `model.` prefix of the module attribute (models.py:408)
    from argparse import Namespace

    from dram_b200.models import ScanRegLightningModule

    module = ScanRegLightningModule(Namespace(model_arch="med3ddram18"))
    utils.load_state_dict_greedy(module, {"model." + k: v for k, v in sd.items()})
    assert float(module.model.layer1[0].conv1.weight.mean()) == 0.5


def test_checkpoint_loading_policy(tmp_path):
    """A Lightning-shaped checkpoint (hyper_parameters Namespace, callbacks, optimizer states — what ModelCheckpoint of
    the reference's train.py writes) loads under torch >= 2.6; a missing file or a Git-LFS pointer is fatal unless
    --allow_random_init."""
    from argparse import Namespace

    from dram_b200 import processor
    from dram_b200.models import ScanRegLightningModule

    module = ScanRegLightningModule(Namespace(model_arch="med3ddram18"))
    sd = {"model." + k: (torch.full_like(v, 0.25) if v.is_floating_point() else v)
          for k, v in module.model.state_dict().items()}
    ckpt = {"epoch": 7, "global_step": 1234, "pytorch-lightning_version": "1.6.4", "state_dict": sd,
            "hyper_parameters": {"args": Namespace(model_arch="med3ddram18", lr=1e-4, target_size=(128, 224, 288))},
            "callbacks": {"ModelCheckpoint{'monitor': 'valid_acc'}": {"best_model_score": torch.tensor(0.5)}},
            "optimizer_states": [{"state": {}, "param_groups": [{"lr": 1e-4}]}], "lr_schedulers": [{"gamma": 0.95}]}
    path = tmp_path / "best.ckpt"
    torch.save(ckpt, path)
    assert processor.load_checkpoint(module, str(path)) is True
    assert float(module.model.layer1[0].conv1.weight.mean()) == 0.25
    # something only the full unpickler accepts (a numpy scalar pickled by an old Lightning): still loads
    ckpt["callbacks"]["x"] = np.float64(1.0)
    torch.save(ckpt, path)
    assert processor.load_checkpoint(module, str(path)) is True
    pointer = tmp_path / "paper.ckpt"
    pointer.write_text("version https://git-lfs.github.com/spec/v1\noid sha256:0\nsize 1\n")
    for bad in (str(pointer), str(tmp_path / "absent.ckpt")):
        with pytest.raises(processor.CheckpointError):
            processor.load_checkpoint(module, bad)
        assert processor.load_checkpoint(module, bad, allow_random_init=True) is False
    assert processor.build_parser().parse_args([]).allow_random_init is False


def test_torch_library_ops_are_registered_with_fake_kernels():
    """north_star: "a thin C-ABI torch custom-op extension" — the dram_b200:: namespace exists, every op has a
    shape-only (fake) kernel so it traces without a GPU, and there is no CPU kernel behind it."""
    from torch._subclasses.fake_tensor import FakeTensorMode

    from dram_b200 import custom_ops, ops  # noqa: F401

    for name in custom_ops.REGISTERED:
        assert hasattr(torch.ops.dram_b200, name), name
    with FakeTensorMode():
        x = torch.empty((2, 8, 10, 12, 64), dtype=torch.float16, device="cuda")
        assert torch.ops.dram_b200.maxpool3d(x).shape == (2, 4, 5, 6, 64)
        assert torch.ops.dram_b200.upsample2x(x).shape == (2, 16, 20, 24, 64)
        w, b = torch.empty((128, 27 * 64), dtype=torch.float16, device="cuda"), torch.empty(128, device="cuda")
        assert torch.ops.dram_b200.conv3d(x, w, b, stride=2).shape == (2, 4, 5, 6, 128)
        assert torch.ops.dram_b200.conv3d(x, w, b, dilation=4).shape == (2, 8, 10, 12, 128)
        img = torch.empty((2, 31, 32, 40), device="cuda")
        sw = torch.empty(28672, dtype=torch.float16, device="cuda")
        assert torch.ops.dram_b200.stem_conv7(img, sw, torch.empty(64, device="cuda")).shape == (2, 16, 16, 20, 64)
        d0 = torch.empty((2, 1, 16, 16, 20), device="cuda")
        m = torch.empty((2, 31, 32, 40), dtype=torch.uint8, device="cuda")
        o0, o1, pct = torch.ops.dram_b200.dram_upsample_mask(d0, d0, m, m)
        assert o0.shape == (2, 1, 31, 32, 40) and pct.shape == (2, 2)
        assert torch.ops.dram_b200.masked_pool(d0, m).shape == (2, 1)
        out, stats = torch.ops.dram_b200.window_standardize(torch.empty((31, 32, 40), dtype=torch.int16, device="cuda"))
        assert out.dtype == torch.float32 and out.shape == (31, 32, 40) and stats.shape == (2,)
        assert torch.ops.dram_b200.heatmap_u8(d0[0, 0], [1, 30, 2, 31, 3, 39], [40, 48, 56]).dtype == torch.uint8
    with pytest.raises(NotImplementedError):
        torch.ops.dram_b200.maxpool3d(torch.zeros(1, 8, 8, 8, 64, dtype=torch.float16))


def test_shard_indices_equal_distributed_sampler():
    from torch.utils.data import DistributedSampler

    from dram_b200.models import shard_indices

    for n in (1, 2, 5, 8, 13):
        for world in (1, 2, 3, 4, 8):
            for rank in range(world):
                ref = list(DistributedSampler(range(n), num_replicas=world, rank=rank, shuffle=False))
                assert shard_indices(n, rank, world) == ref, (n, world, rank)


def test_mha_roundtrip(tmp_path):
    from dram_b200 import mha_io

    rng = np.random.default_rng(0)
    for dtype, compress in ((np.int16, True), (np.uint8, True), (np.float32, False)):
        arr = (rng.standard_normal((5, 7, 9)) * 100).astype(dtype)
        p = str(tmp_path / f"a_{np.dtype(dtype).name}.mha")
        mha_io.write_mha(p, arr, spacing=(0.7, 0.7, 1.25), origin=(-10.0, 3.5, 8.0), compress=compress)
        back, meta = mha_io.read_mha(p)
        assert back.dtype == arr.dtype and np.array_equal(back, arr)
        assert meta["spacing"] == (0.7, 0.7, 1.25) and meta["origin"] == (-10.0, 3.5, 8.0)
        assert meta["direction"] == (1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0)


def test_mha_reader_on_itk_layout_fixtures(tmp_path):
    """Files laid out the way ITK's MetaImageIO writes them (key order, CompressedDataSize, 17-digit doubles,
    TransformMatrix = transposed direction, MSB flag) — built by oracle/make_mha_fixture.py without mha_io — read back
    as sitk.ReadImage + GetArrayFromImage / GetSpacing / GetOrigin / GetDirection would report them
    (dataset.py:49-55), and survive the reference's reversed-rows bookkeeping and our writer."""
    from dram_b200 import mha_io

    with open(os.path.join(GOLDEN, "itk_style_mha.json")) as f:
        expect = json.load(f)
    for name, e in expect.items():
        arr, meta = mha_io.read_mha(os.path.join(GOLDEN, name + ".mha"))
        nx, ny, nz = e["dims_xyz"]
        z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
        want = ((x * 37 + y * 101 + z * 977) % 4096 - 1024).astype(np.int16) if e["kind"] == "int16" \
            else ((x * 7 + y * 13 + z * 29) % 6).astype(np.uint8)
        assert arr.shape == (nz, ny, nx) and arr.dtype == want.dtype and np.array_equal(arr, want), name
        assert meta["spacing"] == tuple(e["spacing"]) and meta["origin"] == tuple(e["origin"]), name
        assert np.allclose(meta["direction"], e["direction"], rtol=0, atol=1e-15), name
        # dataset.py:51-53 reverses to z-y-x, processor.py:146-158 reverses back before writing
        rev = np.asarray(meta["direction"]).reshape(3, 3)[::-1].flatten().tolist()
        back = np.asarray(rev).reshape(3, 3)[::-1].flatten().tolist()
        out = str(tmp_path / (name + "_copy.mha"))
        mha_io.write_mha(out, arr, spacing=meta["spacing"], origin=meta["origin"], direction=back)
        arr2, meta2 = mha_io.read_mha(out)
        assert np.array_equal(arr2, arr) and meta2 == meta, name
    # the header our writer emits has ITK's keys in ITK's order
    with open(out, "rb") as f:
        head = f.read().split(b"ElementDataFile")[0].decode("ascii")
    with open(os.path.join(GOLDEN, "itk_style_ct_oblique.mha"), "rb") as f:
        itk_head = f.read().split(b"ElementDataFile")[0].decode("ascii")
    keys = lambda text: [ln.split("=")[0].strip() for ln in text.strip().splitlines()]  # noqa: E731
    assert [k for k in keys(itk_head)] == [k for k in keys(head)] + ([] if "CompressedDataSize" in head else [])


def test_labels_and_result_merging(tmp_path):
    from argparse import Namespace

    from dram_b200 import processor
    from dram_b200.models import CLE_RATIO_MAP, PSE_RATIO_MAP, ratio_to_label

    with open(os.path.join(GOLDEN, "labels.json")) as f:
        fix = json.load(f)
    ratios = torch.tensor(fix["ratios"], dtype=torch.float32)
    assert [ratio_to_label(r.item(), CLE_RATIO_MAP) for r in ratios] == fix["cle"]
    assert [ratio_to_label(r.item(), PSE_RATIO_MAP) for r in ratios] == fix["pse"]
    rec = lambda uid, s: {"entity": uid, "error_messages": [], "metrics": {  # noqa: E731
        "cle_severity_score": str(s), "cle_lesion_percentage_per_lung": "0.120",
        "pse_severity_score": "1", "pse_lesion_percentage_per_lung": "0.020"}}
    args = Namespace(output_path=str(tmp_path))
    merged = processor.write_results(args, [rec("b", 3), rec("a", 2), rec("b", 3)])  # wrap-around duplicate dropped
    assert [r["entity"] for r in merged] == ["a", "b"]
    assert json.load(open(tmp_path / "centrilobular-emphysema-score.json")) == {"score": 2, "percentage": 0.12}
    assert json.load(open(tmp_path / "araseptal-emphysema-score.json")) == {"score": 1, "percentage": 0.02}
    assert len(json.load(open(tmp_path / "results.json"))) == 2


def test_cli_surface():
    from dram_b200 import processor

    args, extra = processor.build_parser().parse_known_args(
        ["--scan_path", "/a", "--lobe_path", "/b", "--output_path", "/c", "--ngpus", "8", "--target_size", "64,96,128",
         "--accelerator", "gpu", "--max_epochs", "3"])
    assert (args.scan_path, args.lobe_path, args.output_path, args.ngpus) == ("/a", "/b", "/c", 8)
    assert args.target_size == (64, 96, 128) and args.model_arch == "med3ddram" and args.batch_size == 2
    assert extra == ["--accelerator", "gpu", "--max_epochs", "3"]
    assert processor.build_parser().parse_args([]).target_size == (128, 224, 288)


GLOO_WORKER = r"""
import os, sys, json
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
import dram_b200
from dram_b200.models import shard_indices
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
mine = shard_indices(5, rank, world)
gathered = [None] * world
dist.all_gather_object(gathered, mine)
t = torch.tensor([float(rank + 1)], dtype=torch.float64)
dist.all_reduce(t, op=dist.ReduceOp.MAX)          # bench.py's max-over-ranks timing reduction
dist.barrier()
if rank == 0:
    print(json.dumps({"shards": gathered, "max": t.item()}))
dist.destroy_process_group()
"""


def test_two_rank_sharding_over_gloo(tmp_path):
    """World-size-2 run of the multi-GPU host logic on CPU (gloo): every volume lands on exactly one rank
    (plus the wrap-around pad), and the max-over-ranks reduction bench.py times with works."""
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29653", str(script), ROOT],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert res["shards"] == [[0, 2, 4], [1, 3, 0]] and res["max"] == 2.0
    assert set(sum(res["shards"], [])) == set(range(5))


def test_grow_bbox_equals_reference_find_crops():
    """dataset.grow_bbox (host half of row f1) == utils.find_crops of the reference (oracle restatement)."""
    import numpy as np

    from dram_b200.dataset import grow_bbox
    from oracle import pipeline_oracle as P

    rng = np.random.default_rng(0)
    for spacing in [(1.0, 1.0, 1.0), (2.5, 0.7, 0.7), (0.5, 3.0, 1.3)]:
        mask = np.zeros((30, 40, 50), bool)
        lo = rng.integers(0, 10, 3)
        hi = lo + rng.integers(1, 20, 3)
        mask[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = True
        nz = np.nonzero(mask)
        bbox = [v for ax in range(3) for v in (nz[ax].min(), nz[ax].max() + 1)]
        want = [(s.start, s.stop) for s in P.find_crops(mask, spacing, 5)]
        assert grow_bbox(bbox, mask.shape, spacing, 5) == want
        assert grow_bbox(bbox, mask.shape, spacing, 0) == [(bbox[0], bbox[1]), (bbox[2], bbox[3]), (bbox[4], bbox[5])]


GRAD_BUCKET_WORKER = r'''
import json, os, sys
sys.path.insert(0, sys.argv[1])
import torch
import torch.distributed as dist
import dram_b200
from dram_b200.backward import GradBuckets

dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
shapes = [("fcs.0.weight", (1, 32, 1, 1, 1)), ("us3.0.weight", (32, 64, 3, 3, 3)), ("layer1.0.conv1.weight", (64, 64, 3, 3, 3)),
          ("conv1.weight", (64, 1, 7, 7, 7))]
b = GradBuckets(shapes, torch.device("cpu"), bucket_bytes=200000)
for i, (name, shape) in enumerate(shapes):
    b.view(name).fill_(float((rank + 1) * (i + 1)))
for i in range(b.num_buckets):
    b.reduce_bucket(i)
b.wait()
want = [(1 + 2) / 2.0 * (i + 1) for i in range(len(shapes))]
ok = all(bool((b.view(n) == w).all()) for (n, _), w in zip(shapes, want))
if rank == 0:
    print(json.dumps({"ok": ok, "buckets": b.num_buckets, "numel": b.flat.numel(), "bounds": b.bounds}))
dist.destroy_process_group()
'''


def test_gradient_buckets_average_over_two_ranks_gloo(tmp_path):
    """Host logic of the data-parallel exchange (training.TrainStep / backward.GradBuckets) at world size 2 on CPU:
    views alias the flat buffer, buckets close at the byte threshold, every bucket is averaged over the ranks."""
    script = tmp_path / "bucket_worker.py"
    script.write_text(GRAD_BUCKET_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29671", str(script), ROOT],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert res["ok"] and res["buckets"] == 3, res
    assert res["numel"] == 32 + 32 * 64 * 27 + 64 * 64 * 27 + 64 * 343


def test_dgrad_weight_packing_is_the_transposed_flipped_filter():
    """pack_dgrad_weight (CPU-side logic of the data gradient): conv3d(dy, W') with W' = flipped, channel-transposed W
    equals conv_transpose3d(dy, W) — checked with torch on CPU, including a channel slice of a concatenated input."""
    import torch.nn.functional as F

    from dram_b200.backward import pack_dgrad_weight

    g = torch.Generator().manual_seed(0)
    w = torch.randn((64, 128, 3, 3, 3), generator=g)
    dy = torch.randn((1, 64, 5, 6, 7), generator=g)
    for dil, rng in ((1, None), (2, (64, 128))):
        packed = pack_dgrad_weight(w, dtype=torch.float32, cin_range=rng)  # [Cin, 27 * Cout], tap-major
        cin = packed.shape[0]
        wt = packed.view(cin, 3, 3, 3, 64).permute(0, 4, 1, 2, 3)
        got = F.conv3d(dy, wt, None, 1, dil, dil)
        ref = F.conv_transpose3d(dy, w, None, 1, dil, 0, 1, dil)
        ref = ref if rng is None else ref[:, rng[0]:rng[1]]
        assert torch.allclose(got, ref, rtol=1e-4, atol=1e-4)


def test_train_step_flat_layout_and_gradient_routing():
    """Host logic of `training.TrainStep` (no kernel runs): every parameter becomes a view of one flat fp32 buffer with
    its `.grad` at the same offset of the flat gradient buffer, values and `state_dict()` unchanged; convolution weights
    (except the stem and the 1x1x1 heads) and BatchNorm weight/bias pairs are routed to gradient sinks, everything else
    to post-accumulate hooks; bucket counters add up to the parameter count."""
    from dram_b200 import med3d, training

    model = med3d.resnet18segreg().train()
    before = {k: v.clone() for k, v in model.state_dict().items()}
    step = training.TrainStep(model, optimizer="torch", loss="aten", bucket_bytes=16 << 20)
    after = model.state_dict()
    assert list(after) == list(before) and all(torch.equal(before[k], after[k]) for k in before)
    total = sum(p.numel() for p in model.parameters())
    assert step.flat_param.numel() == step.buckets.flat.numel() == total
    for name, p in model.named_parameters():
        off = step.buckets.slices[name][0]
        assert p.data_ptr() == step.flat_param.data_ptr() + 4 * off, name
        assert p.grad.data_ptr() == step.buckets.flat.data_ptr() + 4 * off and p.grad.shape == p.shape, name
    convs = [n for n, m in model.named_modules() if isinstance(m, torch.nn.Conv3d)]
    sinks = sorted(n for n, lay in step.net.layers.items() if lay.grad_sink is not None)
    assert sinks == sorted(n for n in convs if n != "conv1" and not n.startswith("fcs."))
    bns = [m for m in model.modules() if isinstance(m, torch.nn.BatchNorm3d)]
    assert len(step.net.bn_sinks) == len(bns) == 22
    for bn in bns:  # one [dbeta | dgamma] view covering bias.grad then weight.grad
        view, _ = step.net.bn_sinks[id(bn)]
        assert view.data_ptr() == bn.bias.grad.data_ptr() and view.numel() == 2 * bn.num_features
        assert bn.weight.grad.data_ptr() == view.data_ptr() + 4 * bn.num_features
    hooked = sorted(n for n, p in model.named_parameters() if p._post_accumulate_grad_hooks)
    assert hooked == sorted(["conv1.weight", "fcs.0.weight", "fcs.0.bias", "fcs.1.weight", "fcs.1.bias", "us3.0.bias"] +
                            [f"us{i}.conv_blocks.{j}.0.bias" for i in (1, 2) for j in (0, 1)])
    assert sum(step._bucket_size) == len(list(model.parameters())) and step.buckets.num_buckets >= 2
    # a bucket is handed to the exchange exactly when its last gradient has been reported
    fired = []
    step.buckets.reduce_bucket = lambda i, group=None: fired.append(i)
    for b, size in enumerate(step._bucket_size):
        for k in range(size):
            assert fired.count(b) == 0
            step._grad_ready(b)
        assert fired.count(b) == 1
    with pytest.raises(ValueError, match="sync_bn"):
        training.TrainStep(med3d.resnet18segreg().train(), optimizer="torch", loss="aten", sync_bn="maybe")
    with pytest.raises(ValueError, match="loss="):
        training.TrainStep(med3d.resnet18segreg().train(), optimizer="sgd")


def test_conv_descriptor_mirror_matches_the_header():
    """`_capi.ConvDesc` (and the mirror shown in INTEGRATION.md) lists the fields of `dram_conv_desc` in the header's
    order with the header's types — the struct crosses the C-ABI by value layout, so a drift would corrupt every plan."""
    import ctypes as C

    from dram_b200 import _capi

    header = open(os.path.join(ROOT, "include", "dram_b200.h")).read()
    body = header[header.index("typedef struct dram_conv_desc {"):header.index("} dram_conv_desc;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in re.findall(r"int32_t\s+([^;]+);", body):
        for name in decl.split(","):
            name = name.strip()
            m = re.match(r"(\w+)\[(\d+)\]", name)
            fields.append((m.group(1), int(m.group(2))) if m else (name, 1))
    mirror = [(n, t._length_ if hasattr(t, "_length_") else 1) for n, t in _capi.ConvDesc._fields_]
    assert mirror == fields, (mirror, fields)
    assert C.sizeof(_capi.ConvDesc) == 4 * sum(k for _, k in fields)
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = doc[doc.index("class ConvDesc(C.Structure)"):]
    block = block[:block.index("\n\n")]
    doc_fields = [w for lit in re.findall(r'"([a-z0-9_ ]+)"', block) for w in lit.split()]
    assert doc_fields == [n for n, _ in fields], doc_fields


def test_ctypes_signatures_follow_the_header_prototypes():
    """Every entry of `_capi.SIGNATURES` has the arity and return type of its prototype in include/dram_b200.h, and
    pointer / integer / floating-point parameters sit in the same positions (a drifted ctypes signature reads garbage
    off the stack without failing)."""
    import ctypes as C

    from dram_b200 import _capi

    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dram_b200.h")).read(), flags=re.S)
    protos = re.findall(r"\n(int|int64_t|size_t)\s+(dram_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", header)
    assert len(protos) == len(_capi.SIGNATURES), (len(protos), len(_capi.SIGNATURES))
    ret = {"int": C.c_int, "int64_t": C.c_int64, "size_t": C.c_size_t}
    ints = {C.c_int, C.c_int32, C.c_int64, C.c_uint64, C.c_size_t}
    floats = {C.c_float, C.c_double}
    for rtype, name, params in protos:
        res, args = _capi.SIGNATURES[name]
        assert res is ret[rtype], name
        plist = [] if params.strip() in ("", "void") else [p.strip() for p in params.split(",")]
        assert len(plist) == len(args), (name, len(plist), len(args))
        for i, (p, a) in enumerate(zip(plist, args)):
            if "*" in p or "[" in p:
                kind = "pointer"
            elif re.match(r"(const\s+)?(float|double)\b", p):
                kind = "float"
            else:
                kind = "int"
            if kind == "pointer":
                assert a in (C.c_void_p, C.c_char_p) or hasattr(a, "contents") or issubclass(a, C._Pointer), (name, i, p, a)
            elif kind == "float":
                assert a in floats and (a is C.c_double) == ("double" in p), (name, i, p, a)
            else:
                assert a in ints, (name, i, p, a)
                assert (C.sizeof(a) == 8) == bool(re.search(r"u?int64_t|size_t", p)), (name, i, p, a)


def test_built_library_uses_tensor_cores_and_tma():
    """Binary-level check (cuobjdump, no GPU): every convolution kernel that ships in libdram_b200.so issues tcgen05
    MMAs (SASS `UTCHMMA`), reads its accumulators back from tensor memory (`LDTM`) and is fed by TMA (`UTMALDG`; the
    stem stages its operand itself), the staged-epilogue variants store through TMA (`UTMASTG`), and the peer
    exchange kernel carries system-scope release/acquire accesses."""
    import shutil

    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not installed")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_summary
    finally:
        sys.path.pop(0)
    table = sass_summary.kernels()
    tensor = [n for n in table if re.match(r"dram::(conv3d_|upsample2x_umma)", n)]
    assert len(tensor) >= 19, tensor
    for name in tensor:
        c = table[name]
        assert c["UTCHMMA"] > 0 and c["LDTM"] > 0 and c["UTCBAR"] > 0 and c["SYNCS"] > 0, (name, c)
        if "conv3d_stem_kernel" not in name:
            assert c["UTMALDG"] > 0, (name, c)
    for name in ("dram::conv3d_umma_kernel<128, true>", "dram::conv3d_umma_kernel<64, true>", "dram::upsample2x_umma_kernel"):
        assert table[name]["UTMASTG"] > 0, name
    peer = sass_summary.kernel_sass()["dram::peer_allreduce_f64_kernel"]
    for mnemonic in (r"STG\.E\.64\.STRONG\.SYS", r"LDG\.E\.64\.STRONG\.SYS", r"MEMBAR\.SC\.SYS"):
        assert re.search(mnemonic, peer), mnemonic  # st.release.sys flag, ld.acquire.sys poll, __threadfence_system


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly one JSON line on stdout
    with the contract's keys, this run's `cpu_baseline` and a zero-copy `e2e`; under torchrun only rank 0 prints."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "32", "--steps", "2", "--warmup", "1"]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "volumes/s" and line["higher_is_better"] is True
    assert line["steps"] == 2 and line["warmup"] == 1 and line["vs_baseline"] is None and line["data"] == "synthetic"
    assert line["value"] > 0 and abs(line["value"] * line["ms_per_step"] / 1e3 - 1.0) < 1e-6  # one volume per step
    assert "workload" in line["config"] and "32" in line["config"]["workload"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    other = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path), timeout=600, env=env)
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_bench_dump_outputs_budget_and_sample(tmp_path):
    """`bench.py --dump-outputs`: float32 (float64 kept) .npy per output, at most 64 MB in all, arrays too large for
    their share written as the same seeded sample on every run; bad arguments are refused before any work."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    # every map holds its own flat index (exact in float32 below 2^24), so a sample shows which voxels it took
    shape = (2, 1, 160, 160, 160)
    n = int(np.prod(shape))
    g = torch.Generator().manual_seed(0)
    arrays = {"cle_dense_outs": torch.arange(n, dtype=torch.float32).reshape(shape),
              "pse_dense_outs": torch.arange(n, dtype=torch.float64).reshape(shape),
              "cle_precentages": torch.rand(2, generator=g).half(), "pse_precentages": torch.rand(2, generator=g).double()}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(f"{k}.npy" for k in arrays)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    loaded = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert np.array_equal(loaded[f[:-4]], np.load(tmp_path / "b" / f))
    assert loaded["pse_precentages"].dtype == np.float64 and np.array_equal(loaded["pse_precentages"], arrays["pse_precentages"].numpy())
    assert loaded["cle_precentages"].dtype == np.float32
    assert np.array_equal(loaded["cle_precentages"], arrays["cle_precentages"].float().numpy())
    for k, dtype in (("cle_dense_outs", np.float32), ("pse_dense_outs", np.float64)):
        s = loaded[k]
        assert s.dtype == dtype and s.ndim == 1 and 0 < s.size < n, (k, s.dtype, s.shape)
        assert np.array_equal(s, np.round(s)) and s[0] >= 0 and s[-1] < n  # values of the array, i.e. voxel indices
        assert (np.diff(s) > 0).all()                                      # distinct voxels in flat order
        assert s[0] < n // 100 and s[-1] > n - n // 100                    # spread over the whole map
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "c")]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bad, capture_output=True, text=True,
                             cwd=str(tmp_path), timeout=600)
        assert res.returncode == 2 and res.stdout == "", (bad, res.stderr[-500:])
    assert not (tmp_path / "c").exists()


def test_inference_dataset_has_no_cpu_path(tmp_path):
    """Without a CUDA device the dataset reads the files and then refuses: the pre-steps of dataset.py:66-83 exist on
    the GPU only (their CPU restatement is the oracle's, not the product's)."""
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present: the GPU path would run (covered by the -m gpu tests)")
    from dram_b200 import mha_io
    from dram_b200.dataset import SubtypingInference

    (tmp_path / "ct").mkdir()
    (tmp_path / "lobes").mkdir()
    scan = np.full((6, 8, 10), -800, dtype=np.int16)
    lobe = np.zeros((6, 8, 10), dtype=np.uint8)
    lobe[2:4, 2:6, 3:7] = 1
    mha_io.write_mha(str(tmp_path / "ct" / "a.mha"), scan)
    mha_io.write_mha(str(tmp_path / "lobes" / "a.mha"), lobe)
    ds = SubtypingInference(str(tmp_path / "ct"), str(tmp_path / "lobes"))
    assert len(ds) == 1
    with pytest.raises(RuntimeError, match="no CPU path"):
        ds[0]


def test_background_writer_and_read_ahead(tmp_path):
    """`--workers N` of the processor (processor.py:59): the output side writes .mha files on N threads with the same
    bytes as in-place writes and reports a failed write; the input side reads ahead on N threads and hands the loop
    the same batches, in the same order, as the synchronous loader — for full, ragged and wrap-around-padded shards."""
    from argparse import Namespace

    from dram_b200 import mha_io
    from dram_b200.models import SubtypeDataModule

    g = np.random.default_rng(3)
    vols = [(g.integers(0, 4, size=(20, 64, 64)) * 60).astype(np.uint8) for _ in range(6)]
    for sub in ("sync", "async"):
        (tmp_path / sub).mkdir()
    for i, v in enumerate(vols):
        mha_io.write_mha(str(tmp_path / "sync" / f"v{i}.mha"), v, spacing=(0.7, 0.7, 1.25))
    with mha_io.BackgroundWriter(3) as writer:
        for i, v in enumerate(vols):
            writer.submit(mha_io.write_mha, str(tmp_path / "async" / f"v{i}.mha"), v, spacing=(0.7, 0.7, 1.25))
            assert len(writer.pending) <= 6
    for i in range(6):
        assert (tmp_path / "sync" / f"v{i}.mha").read_bytes() == (tmp_path / "async" / f"v{i}.mha").read_bytes()
    writer = mha_io.BackgroundWriter(2)
    writer.submit(mha_io.write_mha, str(tmp_path / "missing_dir" / "x.mha"), vols[0])
    with pytest.raises(FileNotFoundError):
        writer.close()
    inline = mha_io.BackgroundWriter(0)
    inline.submit(mha_io.write_mha, str(tmp_path / "inline.mha"), vols[1])
    assert (tmp_path / "inline.mha").exists() and not inline.pending
    inline.close()

    class FakeDataset:  # stands in for SubtypingInference: file half on the worker threads, device half in the loop
        def __init__(self, n):
            self.n, self.processed = n, []

        def __len__(self):
            return self.n

        def load_raw(self, index):
            return {"uid": f"scan{index:02d}", "value": index}

        def get_data(self, index, raw=None):
            raw = self.load_raw(index) if raw is None else raw
            assert raw["value"] == index
            self.processed.append(index)
            return {"image": torch.full((2, 2), float(index)), "uid": raw["uid"]}

        def __getitem__(self, index):
            return self.get_data(index)

    for n, bs, workers, rank, world in [(7, 2, 3, 0, 1), (7, 3, 1, 1, 2), (5, 4, 8, 2, 3), (1, 2, 2, 0, 1), (4, 2, 2, 3, 4)]:
        batches = {}
        for w in (0, workers):
            dm = SubtypeDataModule(Namespace(batch_size=bs, workers=w, target_size=(8, 8, 8)))
            fake = FakeDataset(n)
            dm.predict_dataset = lambda fake=fake: fake
            batches[w] = [(b["uid"], b["image"][:, 0, 0].tolist()) for b in dm.predict_dataloader(rank, world)]
            from dram_b200.models import shard_indices
            assert fake.processed == shard_indices(n, rank, world)  # the device half runs in order, once per slot
        assert batches[0] == batches[workers] and len(batches[0]) == -(-len(shard_indices(n, rank, world)) // bs)


def test_gpu_cpu_binding_is_optional(monkeypatch):
    """`utils.bind_to_gpu_cpus` (one process per GPU: pinned buffers on the GPU's NUMA node) never raises: without
    NVML / a GPU it reports None and leaves the affinity alone; DRAM_B200_NUMA=0 turns it off."""
    from dram_b200.utils import bind_to_gpu_cpus

    before = os.sched_getaffinity(0)
    res = bind_to_gpu_cpus(0)
    assert res is None or isinstance(res, str)
    if res is None:
        assert os.sched_getaffinity(0) == before
    os.sched_setaffinity(0, before)
    monkeypatch.setenv("DRAM_B200_NUMA", "0")
    assert bind_to_gpu_cpus(0) is None
    assert os.sched_getaffinity(0) == before

