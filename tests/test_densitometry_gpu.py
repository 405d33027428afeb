"""Lung and per-lobe densitometry on the GPU: label counts, HU histograms and HU sums bit-exact against the numpy oracle
(ragged shapes, unaligned views, labels up to 255, more than 16 labels, HU beyond both clamps, absent labels),
reproducibility, guard bands, the custom ops under opcheck and CUDA-graph capture, the processor CLI with
--densitometry, and one full-size scan."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import densitometry_oracle as O
from oracle import synthetic

pytestmark = pytest.mark.gpu

SHAPES = [(63, 67, 250), (16, 16, 17), (64, 64, 64), (5, 7, 3)]
CASES = ["lobes", "palette", "many_labels", "background_tracked"]


def _volume(shape, case, seed=0):
    """(scan int16, labels uint8, label ids to histogram) on the CPU."""
    g = torch.Generator().manual_seed(seed)
    scan, labels = synthetic.make_volume(70 + seed, shape)
    lung = torch.nonzero(labels.reshape(-1) > 0).reshape(-1)
    if lung.numel() >= 2:   # HU beyond both clamps inside a lobe
        scan.view(-1)[lung[0]] = -3024
        scan.view(-1)[lung[-1]] = 3071
    ids = [1, 2, 3, 4, 5, 9]                                    # 9: an absent label
    if case == "palette":
        palette = torch.tensor([0, 1, 2, 7, 200, 255], dtype=torch.uint8)
        labels = palette[torch.randint(0, len(palette), shape, generator=g)]
        ids = [255, 1, 2, 7, 200, 3]
    elif case == "many_labels":                                 # three passes of up to 16 labels
        labels = torch.randint(0, 40, shape, generator=g, dtype=torch.uint8)
        ids = list(range(1, 40))
    elif case == "background_tracked":                          # label 0 tracked too: every vector reads its HU
        ids = [0, 3, 5]
    return scan, labels, ids


def _check(scan, labels, ids, counts, hist, sums):
    assert counts.dtype == hist.dtype == sums.dtype == torch.int64
    assert np.array_equal(counts.cpu().numpy(), O.label_counts(labels.numpy())), "label counts differ"
    ref_hist, ref_sums = O.hu_histograms(scan.numpy(), labels.numpy(), ids)
    assert np.array_equal(hist.cpu().numpy(), ref_hist), "histograms differ"
    assert np.array_equal(sums.cpu().numpy(), ref_sums), "HU sums differ"


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("shape", SHAPES)
def test_counts_and_histograms_bit_exact_and_repeatable(cuda, lib, shape, case):
    from dram_b200 import ops

    scan, labels, ids = _volume(shape, case)
    s, lab = scan.to(cuda), labels.to(cuda)
    counts = ops.label_counts(lab)
    hist, sums = ops.hu_histograms(s, lab, ids)
    _check(scan, labels, ids, counts, hist, sums)
    if case == "lobes":
        assert hist[ids.index(9)].sum().item() == 0 and counts[9].item() == 0
    for _ in range(2):
        assert torch.equal(ops.label_counts(lab), counts)
        h2, s2 = ops.hu_histograms(s, lab, ids)
        assert torch.equal(h2, hist) and torch.equal(s2, sums)


@pytest.mark.parametrize("shape", [(63, 67, 250), (16, 16, 17)])
def test_unaligned_views_take_the_byte_path(cuda, lib, shape):
    from dram_b200 import ops

    scan, labels, ids = _volume(shape, "palette", seed=2)
    raw_l = torch.zeros(labels.numel() + 3, dtype=torch.uint8, device=cuda)
    raw_s = torch.zeros(scan.numel() + 1, dtype=torch.int16, device=cuda)
    lab_u, scan_u = raw_l[3:].view(shape), raw_s[1:].view(shape)
    lab_u.copy_(labels.to(cuda))
    scan_u.copy_(scan.to(cuda))
    assert lab_u.data_ptr() % 16 == 3 and scan_u.data_ptr() % 16 == 2
    counts = ops.label_counts(lab_u)
    hist, sums = ops.hu_histograms(scan_u, lab_u, ids)
    _check(scan, labels, ids, counts, hist, sums)
    # aligned labels with an unaligned scan
    hist2, sums2 = ops.hu_histograms(scan_u, labels.to(cuda), ids)
    assert torch.equal(hist2, hist) and torch.equal(sums2, sums)


def test_outputs_stay_inside_their_allocation(cuda, lib):
    """Both calls write their outputs exactly: a sentinel-filled allocation around them stays intact."""
    from dram_b200 import _capi, ops

    PAD = 4096
    scan, labels, ids = _volume((9, 13, 31), "palette", seed=3)
    s, lab = scan.to(cuda), labels.to(cuda)
    n = labels.numel()

    def guarded(numel):
        raw = torch.full((2 * PAD + numel * 8,), 0xA5, dtype=torch.uint8, device=cuda)
        return raw, raw[PAD:PAD + numel * 8].view(torch.int64)

    def intact(raw, nbytes, what):
        torch.cuda.synchronize()
        assert bool((raw[:PAD] == 0xA5).all()) and bool((raw[PAD + nbytes:] == 0xA5).all()), what

    raw_c, counts = guarded(256)
    _capi.check(lib.dram_label_counts(ops._p(lab), n, ops._p(counts), ops._stream()), "dram_label_counts")
    intact(raw_c, 256 * 8, "label counts")
    nslots = 5
    table = bytearray(b"\xff" * 256)
    for i, k in enumerate(ids[:nslots]):
        table[k] = i
    raw_h, hist = guarded(nslots * 2048)
    raw_s, sums = guarded(nslots)
    _capi.check(lib.dram_label_hu_hist(ops._p(s), ops._p(lab), n, bytes(table), nslots, ops._p(hist), ops._p(sums),
                                       ops._stream()), "dram_label_hu_hist")
    intact(raw_h, nslots * 2048 * 8, "histograms")
    intact(raw_s, nslots * 8, "HU sums")
    _check(scan, labels, ids[:nslots], counts, hist.view(nslots, 2048), sums)


def test_ops_opcheck_and_graph_capture(cuda, lib):
    from dram_b200 import ops

    scan, labels, ids = _volume((16, 24, 32), "lobes", seed=4)
    s, lab = scan.to(cuda), labels.to(cuda)
    torch.library.opcheck(torch.ops.dram_b200.label_counts.default, (lab,))
    torch.library.opcheck(torch.ops.dram_b200.hu_histograms.default, (s, lab, ids))
    assert torch.equal(torch.ops.dram_b200.label_counts(lab), ops.label_counts(lab))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gc = torch.ops.dram_b200.label_counts(lab)
        gh, gs = torch.ops.dram_b200.hu_histograms(s, lab, ids)
    new_scan, new_labels, _ = _volume((16, 24, 32), "palette", seed=8)
    s.copy_(new_scan.to(cuda))
    lab.copy_(new_labels.to(cuda))
    graph.replay()
    torch.cuda.synchronize()
    _check(new_scan, new_labels, ids, gc, gh, gs)


def test_scan_densitometry_equals_the_oracle(cuda, lib):
    from dram_b200 import densitometry

    spacing = (1.25, 0.7, 0.7)
    for case in ("lobes", "many_labels"):
        scan, labels, _ = _volume((40, 48, 56), case, seed=5)
        got = densitometry.scan_densitometry(scan.to(cuda), labels.to(cuda), spacing)
        assert got == O.densitometry(scan.numpy(), labels.numpy(), spacing)


def _write_scans(tmp_path, scan_dims, label_dtype):
    from dram_b200 import mha_io

    scan_dir, lobe_dir = tmp_path / "ct", tmp_path / "lobes"
    scan_dir.mkdir(exist_ok=True)
    lobe_dir.mkdir(exist_ok=True)
    for i in range(3):
        ct, lobes = synthetic.make_volume(40 + i, scan_dims)
        inside = torch.nonzero(lobes.reshape(-1) == 2).reshape(-1)
        ct.view(-1)[inside[:5]] = -3024
        ct.view(-1)[inside[-5:]] = 3071
        kw = dict(spacing=(0.7, 0.7, 1.25), origin=(1.0, 2.0, 3.0))   # x, y, z: 1.25 mm slices
        mha_io.write_mha(str(scan_dir / f"scan{i}.mha"), ct.numpy(), **kw)
        mha_io.write_mha(str(lobe_dir / f"scan{i}.mha"), lobes.numpy().astype(label_dtype), **kw)
    return scan_dir, lobe_dir


def _run(argv_base, out_dir, extra=()):
    from dram_b200 import processor

    records = processor.run_testing_job(argv_base + ["--output_path", str(out_dir)] + list(extra))
    files = {}
    for root, _, names in os.walk(out_dir):
        for f in names:
            if f != "results.json":
                files[os.path.relpath(os.path.join(root, f), out_dir)] = open(os.path.join(root, f), "rb").read()
    return records, files, open(out_dir / "results.json", "rb").read()


@pytest.mark.parametrize("arch,workers,label_dtype", [("med3ddram18", 0, np.uint8), ("med3ddram18", 2, np.int16),
                                                      ("med3d18", 0, np.int16), ("med3d18", 2, np.uint8)])
def test_processor_densitometry_end_to_end(cuda, lib, tmp_path, arch, workers, label_dtype):
    from dram_b200 import densitometry, mha_io

    scan_dir, lobe_dir = _write_scans(tmp_path, (40, 48, 56), label_dtype)
    target = "32,40,48" if "dram" in arch else "64,64,64"
    sd = synthetic.make_state_dict(arch, seed=7, calib_dims=tuple(int(v) for v in target.split(",")), prefix="model.")
    ckpt = tmp_path / "best.ckpt"
    torch.save({"state_dict": sd}, ckpt)
    argv = ["--scan_path", str(scan_dir), "--lobe_path", str(lobe_dir), "--model_arch", arch, "--target_size", target,
            "--batch_size", "2", "--ckpt_path", str(ckpt), "--workers", str(workers)]
    plain, files_plain, _ = _run(argv, tmp_path / "plain")
    got, files_got, _ = _run(argv, tmp_path / "dens", ["--densitometry"])
    assert files_got == files_plain, "heat-maps or score files changed with --densitometry"
    assert [{k: v for k, v in r.items() if k != "densitometry"} for r in got] == plain
    assert all("densitometry" not in r for r in plain)
    on_disk = json.load(open(tmp_path / "dens" / "results.json"))
    assert on_disk == got and len(got) == 3
    for rec in got:
        scan, meta = mha_io.read_mha(str(scan_dir / f"{rec['entity']}.mha"))
        lobes, _ = mha_io.read_mha(str(lobe_dir / f"{rec['entity']}.mha"))
        assert lobes.dtype == label_dtype
        want = densitometry.format_densitometry(O.densitometry(scan, lobes, meta["spacing"][::-1]))
        assert rec["densitometry"] == want, rec["entity"]
        assert sorted(rec["densitometry"]["lobes"]) == ["1", "2", "3", "4", "5"]


def test_full_size_scan(cuda, lib):
    """One 400 x 512 x 512 scan: counts, histograms and the measures against the oracle."""
    from dram_b200 import densitometry, ops

    dims, spacing = (400, 512, 512), (1.0, 0.68, 0.68)
    scan, labels = synthetic.make_volume(11, dims)
    s, lab = scan.to(cuda), labels.to(cuda)
    got = densitometry.scan_densitometry(s, lab, spacing)
    ids = [1, 2, 3, 4, 5]
    counts = ops.label_counts(lab)
    hist, sums = ops.hu_histograms(s, lab, ids)
    _check(scan, labels, ids, counts, hist, sums)
    assert got == O.densitometry(scan.numpy(), labels.numpy(), spacing)
    print("full-size densitometry:", densitometry.format_densitometry(got)["lung"])
