"""Drop-in `models` module: `ScanRegLightningModule`, `ScanCLSLightningModule`, `SubtypeDataModule`.

Same constructor (`args` namespace with `model_arch`, `target_size`, `scan_path`, ...), same
attributes (`.model`, `.args`) and the same `forward(x, lungs)` / `predict_step(batch, batch_idx)`
contract as models.py:160-181, 397-450 and 36-96 of the reference — the returned dict keeps the
reference's seven keys and their spelling.  If pytorch_lightning is importable the classes derive
from its LightningModule/LightningDataModule; otherwise from light stand-ins with the same surface,
so `processor.py` runs without Lightning (SURVEY H9).

`ScanRegLightningModule` also carries the reference's training surface (`training_step`, `validation_step`,
`test_step`, `configure_optimizers`; models.py:530-600, 685-698) on `training.TrainStep` — manual optimisation: one
call runs forward, loss, backward, the gradient exchange and Adam on the sm_100a kernels.  The classification
module's training and the epoch-end reporting (confusion matrices, CSVs, debug drawings) are not built.
"""
import enum

import torch

from . import ops
from .dataset import SubtypingInference
from .transforms import InferenceTransform
from .utils import get_model_by_name

try:  # pragma: no cover - not installed in the build image
    import pytorch_lightning as pl
    from pytorch_lightning.trainer.states import RunningStage

    _ModuleBase, _DataModuleBase = pl.LightningModule, pl.LightningDataModule
except ImportError:
    class RunningStage(str, enum.Enum):
        TRAINING = "train"
        VALIDATING = "validate"
        TESTING = "test"
        PREDICTING = "predict"

    class _ModuleBase(torch.nn.Module):
        def save_hyperparameters(self, *args, **kwargs):
            pass

    class _DataModuleBase:
        def __init__(self, *args, **kwargs):
            pass

TRAIN_PHASE = RunningStage.TRAINING
VALID_PHASE = RunningStage.VALIDATING
TEST_PHASE = RunningStage.TESTING
PREDICT_PHASE = RunningStage.PREDICTING

CLE_RATIO_MAP = {0: (0.0, 0.01), 1: (0.01, 0.05), 2: (0.05, 0.1), 3: (0.1, 0.2), 4: (0.2, 0.3), 5: (0.3, 1.0001)}
PSE_RATIO_MAP = {0: (0.0, 0.01), 1: (0.01, 0.05), 2: (0.05, 1.0001)}


def ratio_to_label(ratio, ratio_mapping):
    """First bin with lo <= ratio < hi (processor.py:34-38, models.py:533-537); IndexError outside."""
    hits = [label for label, (lo, hi) in ratio_mapping.items() if lo <= ratio and ratio < hi]
    return hits[0]


def _as_u8(mask):
    """bool/uint8 [B,D,H,W] device mask as uint8 without a copy when possible."""
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    if mask.dtype == torch.uint8:
        return mask.contiguous()
    return (mask != 0).to(torch.uint8)


def _lobe_outputs(cle, pse, ess, labels):
    """The per-label keys of predict_step: voxel counts and both lesion percentages of every label 0..255, each
    divided by that label's own voxel count (never the batch-wide denominator of quirk Q1)."""
    pct, voxels = ops.lobe_scores(cle, pse, ess, labels.contiguous())
    return {"lobe_voxels": voxels, "cle_lobe_percentages": pct[0], "pse_lobe_percentages": pct[1]}


class SubtypeDataModule(_DataModuleBase):
    """models.py:36-96 (prediction part): builds `SubtypingInference` with the inference transform."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        self.datasets = {TRAIN_PHASE: TRAIN_PHASE, VALID_PHASE: VALID_PHASE, TEST_PHASE: TEST_PHASE,
                         PREDICT_PHASE: PREDICT_PHASE}

    def _make_transforms(self, mode):
        if mode == TRAIN_PHASE:
            raise NotImplementedError("training augmentations are outside the inference hot path")
        device = getattr(self.args, "device", None)
        return InferenceTransform(tuple(self.args.target_size), device=device)

    def predict_dataset(self):
        self.datasets[PREDICT_PHASE] = SubtypingInference(
            scan_path=self.args.scan_path, lobe_path=self.args.lobe_path,
            transforms=self._make_transforms(TEST_PHASE), lobe_labels=bool(getattr(self.args, "lobe_scores", False)),
            densitometry=bool(getattr(self.args, "densitometry", False)))
        return self.datasets[PREDICT_PHASE]

    def predict_dataloader(self, rank=0, world_size=1):
        """Batches of the rank's shard: index r, r+N, ... of the sorted file list, padded by wrap-around
        to equal length, like DistributedSampler(shuffle=False) (models.py:92)."""
        ds = self.predict_dataset()
        indices = shard_indices(len(ds), rank, world_size)
        bs = int(getattr(self.args, "batch_size", 2))
        workers = int(getattr(self.args, "workers", 0) or 0)
        if workers <= 0:
            for i in range(0, len(indices), bs):
                yield collate([ds[j] for j in indices[i:i + bs]])
            return
        # `--workers N` (processor.py:59, the reference's DataLoader workers): N threads read the .mha files of the
        # scans ahead (file I/O + zlib, GIL released) while the GPU works; the device pre-steps stay in this thread
        from concurrent.futures import ThreadPoolExecutor

        ahead = workers + bs
        with ThreadPoolExecutor(max_workers=workers, thread_name_prefix="mha-read") as pool:
            futures = {}
            for pos in range(len(indices)):
                for q in range(pos, min(pos + ahead, len(indices))):
                    if q not in futures:
                        futures[q] = pool.submit(ds.load_raw, indices[q])
                if pos % bs == 0:
                    samples = []
                samples.append(ds.get_data(indices[pos], raw=futures.pop(pos).result()))
                if len(samples) == bs or pos == len(indices) - 1:
                    yield collate(samples)

    def train_dataloader(self):
        raise NotImplementedError("training is not part of this build")

    val_dataloader = test_dataloader = train_dataloader


def shard_indices(n, rank, world_size):
    """DistributedSampler(shuffle=False, drop_last=False): pad to a multiple of world_size by repeating
    from the start, then take every world_size-th index starting at `rank`."""
    if n == 0:
        return []
    total = -(-n // world_size) * world_size
    idx = list(range(n))
    while len(idx) < total:
        idx += idx[: total - len(idx)]
    return idx[rank:total:world_size]


def collate(samples):
    """torch's default_collate for the dataset dicts: tensors stacked, strings listed."""
    out = {}
    for key in samples[0]:
        vals = [s[key] for s in samples]
        if isinstance(vals[0], torch.Tensor):
            out[key] = torch.stack(vals)
        elif isinstance(vals[0], str):
            out[key] = list(vals)
        else:
            out[key] = torch.as_tensor(vals)
    return out


class DevicePrefetcher:
    """Wraps an iterable of host batch dicts (the `predict_dataloader` contract, ideally pinned memory):
    the tensors of batch i+1 are copied host->device on side streams while the caller computes on batch
    i.  Two device buffer sets are reused in turn; a set is overwritten only after the compute stream has
    passed the point where the caller asked for the following batch.  Non-tensor entries pass through.

    With `copy_streams` > 1 large tensors are cut into 16 MB chunks that travel on several streams at once.
    Measured A/B on one box (ResNet-34, 256^3, batch 4; profiles/bench_b4_r1o_copy{1,4}.json): one stream 23.7 ms
    per step end to end, four streams 24.5 ms — more DMA engines in flight take a little from the kernels and the
    copy was already hidden — so one stream is the default; the switch is kept for hosts where a single DMA stream
    cannot keep up (one box of this round showed 9 GB/s under load against 47 GB/s idle).

        for batch in DevicePrefetcher(loader, device):
            pred = module.predict_step(batch, i)
    """

    CHUNK_BYTES = 16 << 20

    def __init__(self, loader, device, copy_streams=1):
        self.loader, self.device = loader, torch.device(device)
        self.copy_streams = [torch.cuda.Stream(device=self.device) for _ in range(max(1, int(copy_streams)))]
        self.copy_stream = self.copy_streams[0]

    def _stage(self, host, bufs, done):
        out, pieces = {}, []
        for key, val in host.items():
            if isinstance(val, torch.Tensor) and not val.is_cuda:
                dst = bufs.get(key)
                if dst is None or dst.shape != val.shape or dst.dtype != val.dtype:
                    dst = bufs[key] = torch.empty(val.shape, dtype=val.dtype, device=self.device)
                out[key] = dst
                nbytes = val.numel() * val.element_size()
                if val.is_contiguous() and nbytes > self.CHUNK_BYTES and len(self.copy_streams) > 1:
                    src, flat = val.view(-1), dst.view(-1)
                    step = -(-val.numel() // (-(-nbytes // self.CHUNK_BYTES)))
                    pieces.extend((flat[o:o + step], src[o:o + step]) for o in range(0, val.numel(), step))
                else:
                    pieces.append((dst, val))
            else:
                out[key] = val
        ready = []
        for si, stream in enumerate(self.copy_streams):
            mine = pieces[si::len(self.copy_streams)]
            if not mine:
                continue
            with torch.cuda.stream(stream):
                if done is not None:
                    stream.wait_event(done)
                for d, v in mine:
                    d.copy_(v, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(stream)
                ready.append(ev)
        return out, ready

    def __iter__(self):
        it = iter(self.loader)
        bufs, done = ({}, {}), [None, None]
        try:
            staged = self._stage(next(it), bufs[0], None)
        except StopIteration:
            return
        k = 0
        while staged is not None:
            cur, ready = staged
            try:
                nxt = next(it)
            except StopIteration:
                nxt = None
            # batch k+1 goes into the set batch k-1 used; the caller finished issuing work on k-1 before
            # asking for k, and `done` was recorded on its stream at that moment
            staged = self._stage(nxt, bufs[(k + 1) % 2], done[(k + 1) % 2]) if nxt is not None else None
            for ev in ready:
                torch.cuda.current_stream(self.device).wait_event(ev)
            yield cur
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            done[k % 2] = ev
            k += 1


class _ScanModule(_ModuleBase):
    def __init__(self, args):
        self.args = args
        super().__init__()
        self.model = get_model_by_name(args.model_arch)
        self.save_hyperparameters()
        self.trace = True

    def forward(self, x, lungs):
        return self.model(x, lungs)

    def _unsupported(self, *a, **k):
        raise NotImplementedError("dram_b200 implements the inference path (forward / predict_step) only")

    training_step = validation_step = test_step = configure_optimizers = _unsupported

    def _to_device(self, t):
        dev = next(self.model.parameters()).device
        return t if t.device == dev else t.to(dev, non_blocking=True)


class ScanRegLightningModule(_ScanModule):
    """models.py:397-450.  `per_sample_percentage=True` divides each sample's dRAM sum by its own lung
    volume instead of the whole batch's (reference quirk Q1, models.py:440-441); default = reference."""

    def __init__(self, args):
        super().__init__(args)
        self.beta, self.gamma = 0.7338, 0.2578
        self.per_sample_percentage = bool(getattr(args, "per_sample_percentage", False))

    def predict_step(self, batch, batch_idx, dataloader_idx=0):
        with torch.no_grad():
            image = self._to_device(batch["image"]).float().contiguous()
            lungs = _as_u8(self._to_device(batch["lung_mask"]))
            ess = _as_u8(self._to_device(batch["ess_mask"]))
            if self.model.head_kind != "reg":
                raise RuntimeError(f"{type(self).__name__} needs a *dram (regression) architecture, got a "
                                   "classification one; use ScanCLSLightningModule for med3d/med3d18/med3d50")
            B, D, H, W = image.shape
            eng = self.model.eval().engine(B, (D, H, W), image.device)
            # the lobe-masked means of forward() are not used here (quirk Q2): no K6.  K7 reads the dense maps only
            # around `ess`: the full-resolution decoder runs there only (active_ess)
            if hasattr(eng, "stem_weights"):
                dense = eng.run_network(first=eng.image_stem(image), active_ess=ess)  # the stem reads the image in place
            else:
                eng.load_image(image)
                dense = eng.run_network(active_ess=ess)
            cle, pse, pct = ops.dram_upsample_mask(dense[0], dense[1], ess, lungs, (D, H, W),
                                                   per_sample_denominator=self.per_sample_percentage)
            out = {
                "cle_dense_outs": cle,
                "pse_dense_outs": pse,
                "cle_precentages": pct[0],
                "pse_precentages": pct[1],
                "crop_slices": batch.get("crop_slice"),
                "original_size": batch.get("original_size"),
                "uids": batch.get("uid"),
            }
            if "lobe_labels" in batch:
                out.update(_lobe_outputs(cle, pse, ess, self._to_device(batch["lobe_labels"])))
            return out

    def predict_step_from_hu(self, hu, lung_mask, ess_mask, fuse_window=None, lobe_labels=None):
        """The device-resident hot path of SURVEY §8d: int16 HU volumes already at network size [B,D,H,W] -> K8
        window + standardise (per volume) -> network -> dRAM.  `fuse_window=True`: K8 is its statistics pass plus an
        851-entry table per volume, and the stem convolution clamps and gathers while it loads the int16 volume (the
        same values bit for bit; the fp32 image is never written).  `fuse_window=False`: K8 writes the fp32 image first
        (what predict_step receives from the transforms).  Default (None): env DRAM_B200_FUSE_WINDOW, else False — the
        stem kernel is bound by its producers' instruction issue, and the table gathers cost it more (0.38 against
        0.23 ms per 256^3 volume, profiles/aux_metrics_r2b.csv) than K8's apply pass saves (0.03 ms).  Returns the same dict as predict_step (without the bookkeeping keys).
        `lobe_labels`: optional uint8 [B,D,H,W] label volumes; adds the per-label keys predict_step adds for a batch
        that carries them."""
        with torch.no_grad():
            if not hu.is_cuda or hu.dtype != torch.int16:
                raise RuntimeError("predict_step_from_hu: expected an int16 CUDA tensor [B,D,H,W]")
            B, D, H, W = hu.shape
            eng = self.model.eval().engine(B, (D, H, W), hu.device)
            hu = hu.contiguous()
            if fuse_window is None:
                import os

                fuse_window = os.environ.get("DRAM_B200_FUSE_WINDOW", "0").lower() in ("1", "on", "true", "yes")
            lungs, ess = _as_u8(lung_mask), _as_u8(ess_mask)
            if fuse_window and hasattr(eng, "stem_weights"):
                lut, _ = ops.window_lut(hu)  # statistics are per volume (intensity_transforms.py:104-114)
                dense = eng.run_network(first=eng.hu_stem(hu, lut), active_ess=ess)
            else:
                ops.window_standardize(hu, out=eng.image, batched=True)
                dense = eng.run_network(active_ess=ess)
            cle, pse, pct = ops.dram_upsample_mask(dense[0], dense[1], ess, lungs, (D, H, W),
                                                   per_sample_denominator=self.per_sample_percentage)
            out = {"cle_dense_outs": cle, "pse_dense_outs": pse, "cle_precentages": pct[0],
                   "pse_precentages": pct[1]}
            if lobe_labels is not None:
                out.update(_lobe_outputs(cle, pse, ess, lobe_labels))
            return out

    def _ratio_to_label(self, ratios, ratio_mapping):
        labels = [ratio_to_label(r.item(), ratio_mapping) for r in ratios]
        return torch.as_tensor(labels).long().to(ratios.device)

    # ------------------------------------------------------------------ training surface (SURVEY 8f f4)
    automatic_optimization = False  # under Lightning: training_step does backward + optimiser itself

    def configure_optimizers(self):
        """The reference returns torch.optim.Adam(lr=args.lr) + ExponentialLR(0.95) (models.py:685-698) for Lightning
        to drive; here Adam is K12 inside `training_step` and the decay is `on_train_epoch_end`, so there is nothing
        for the trainer to step."""
        return None

    def _class_weights(self, name, labels):
        table = getattr(self, name, None)
        if table is None:  # models.py:546-551 reads them from the training dataset
            try:
                table = getattr(self.trainer.datamodule.datasets[RunningStage.TRAINING], name)
            except Exception:
                table = None
        if table is None:
            # the reference reads the table from its training dataset and fails without one (models.py:546-551);
            # uniform weights change the loss, so say so once instead of silently training something else
            if not getattr(self, "_warned_class_weights", False):
                import warnings

                warnings.warn(f"{name} not set on the module or its datamodule's training dataset: using uniform class "
                              "weights (the reference raises here)", RuntimeWarning, stacklevel=3)
                object.__setattr__(self, "_warned_class_weights", True)
            return torch.ones(len(labels), dtype=torch.float32)
        return torch.tensor([float(table[int(c)]) for c in labels], dtype=torch.float32)

    def train_engine(self):
        """The `training.TrainStep` behind `training_step` (built on first use; owns the flat parameter, gradient and
        Adam buffers).  Data-parallel when torch.distributed is initialised: gradient all-reduce per bucket and
        SyncBatchNorm, as train.py:100-101 ask of Lightning."""
        eng = getattr(self, "_train_engine", None)
        if eng is None:
            import torch.distributed as dist

            from . import training

            if self.model.head_kind != "reg":
                raise RuntimeError("training_step needs a *dram (regression) architecture (train.py:72)")
            import os

            multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
            sync_bn = False
            if multi:
                # one node with all ranks local (torchrun exports LOCAL_WORLD_SIZE): the statistics travel over NVLink
                # peer memory (K10x); across nodes NCCL carries them
                local = int(os.environ.get("LOCAL_WORLD_SIZE", "0"))
                sync_bn = "peer" if local == dist.get_world_size() <= 8 else "nccl"
            eng = training.TrainStep(self.model.train(), lr=float(getattr(self.args, "lr", 1e-4)), sync_bn=sync_bn)
            object.__setattr__(self, "_train_engine", eng)
        return eng

    def training_step(self, batch, batch_idx):
        """shared_step(TRAIN), models.py:530-570: returns the reference's dict (`loss` detached: backward and the
        Adam step already happened) plus the four logged loss terms."""
        from . import training

        dev = next(self.model.parameters()).device
        cle_labels, pse_labels = batch["cls_label"].reshape(-1).long(), batch["pse_label"].reshape(-1).long()
        bands = [training.regression_label_bands(lab.tolist(), table).to(dev)
                 for lab, table in ((cle_labels, CLE_RATIO_MAP), (pse_labels, PSE_RATIO_MAP))]
        weights = [self._class_weights(name, lab.tolist()).to(dev)
                   for name, lab in (("cle_class_weights", cle_labels), ("pse_class_weights", pse_labels))]
        dev_batch = {"image": self._to_device(batch["image"]).float().contiguous(),
                     "lung_mask": self._to_device(batch["lung_mask"]), "em_mask": self._to_device(batch["em_mask"]),
                     "cls_label": cle_labels.to(dev), "pse_label": pse_labels.to(dev)}
        if not self.model.training:
            self.model.train()
        eng = self.train_engine()
        loss = eng.step(dev_batch, bands[0], bands[1], weights[0], weights[1])
        regs = eng.last["reg_outs"]
        out = {"loss": loss, "pred_cle_labels": self._ratio_to_label(regs[0], CLE_RATIO_MAP),
               "pred_pse_labels": self._ratio_to_label(regs[1], PSE_RATIO_MAP),
               "cle_labels": cle_labels, "pse_labels": pse_labels,
               "index": batch["index"].squeeze(-1) if "index" in batch else None}
        out.update({k: v for k, v in eng.last.items() if k != "reg_outs"})
        return out

    def on_train_epoch_end(self):
        eng = getattr(self, "_train_engine", None)
        if eng is not None:
            eng.decay_lr(0.95)  # ExponentialLR(gamma=0.95), one step per epoch (models.py:694-697)
            if eng.peer is not None:
                eng.peer.check()  # a SyncBatchNorm exchange that timed out fell back to local statistics: fail loudly

    # Lightning's checkpoint hooks: the optimiser lives in K12's flat buffers, not in configure_optimizers(), so its
    # state (Adam moments, step count, decayed learning rate) travels in the checkpoint under its own key.
    def on_save_checkpoint(self, checkpoint):
        eng = getattr(self, "_train_engine", None)
        if eng is not None and hasattr(eng.opt, "exp_avg"):
            checkpoint["dram_b200_flat_adam"] = {k: (v.detach().cpu() if isinstance(v, torch.Tensor) else v)
                                                 for k, v in eng.opt.state_dict().items()}

    def on_load_checkpoint(self, checkpoint):
        state = checkpoint.get("dram_b200_flat_adam")
        if state is not None:
            eng = self.train_engine()
            if hasattr(eng.opt, "exp_avg"):
                eng.opt.load_state_dict(state)

    def _eval_step(self, batch, batch_idx):
        """shared_step(VALID / TEST), models.py:571-582 without the debug drawings: forward, predicted labels."""
        with torch.no_grad():
            image = self._to_device(batch["image"]).float()
            lungs = _as_u8(self._to_device(batch["lung_mask"]))
            _, regs = self.model.eval()(image.unsqueeze(1).contiguous(), lungs)
            return {"pred_cle_labels": self._ratio_to_label(regs[0], CLE_RATIO_MAP),
                    "pred_pse_labels": self._ratio_to_label(regs[1], PSE_RATIO_MAP),
                    "cle_labels": batch["cls_label"], "pse_labels": batch["pse_label"],
                    "index": batch["index"].squeeze(-1) if "index" in batch else None}

    validation_step = test_step = _eval_step


class ScanCLSLightningModule(_ScanModule):
    """models.py:160-181; prediction = argmax of the pooled class logits (models.py:245-247)."""

    def predict_step(self, batch, batch_idx, dataloader_idx=0):
        with torch.no_grad():
            image = self._to_device(batch["image"]).float().contiguous()
            if self.model.head_kind != "cls":
                raise RuntimeError(f"{type(self).__name__} needs a classification architecture (med3d*)")
            B, D, H, W = image.shape
            eng = self.model.eval().engine(B, (D, H, W), image.device)
            _, logits = eng.run(image, None)
            return {
                "cle_logits": logits[0].clone(),
                "pse_logits": logits[1].clone(),
                "cle_labels": logits[0].argmax(-1),
                "pse_labels": logits[1].argmax(-1),
                "crop_slices": batch.get("crop_slice"),
                "original_size": batch.get("original_size"),
                "uids": batch.get("uid"),
            }
