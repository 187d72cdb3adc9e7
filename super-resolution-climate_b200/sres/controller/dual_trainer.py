"""ModelTrainer, mirror of sres/controller/dual_trainer.py:110-571 for the tile path.

Same public methods and return shapes as the reference controller API (SURVEY.md 8b):
  train, evaluate, process_image, apply_network, loss, assemble_images (+ denorm, ttsplit_times).
Differences are confined to where the work runs: batches stay on the GPU from tile extraction to
stitching, the model / loss / optimizer are the CUDA kernels, and under torchrun the tile batches of a
timeslice are sharded across ranks with the gradient all-reduce overlapped with backward.
"""
import ctypes as C
import random
import time
from typing import Any, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.distributed as dist
from torch import Tensor

from sres.base.gpu import set_device
from sres.base.util.array import array2tensor, downsample, upsample
from sres.base.util.config import ConfigContext, cfg
from sres.controller.checkpoints import CheckpointManager
from sres.controller.config import TSet
from sres.data.batch import BatchDataset, TileArray
from sres.data.tiles import TileIterator
from sres.model.manager import SRModels
from sres_b200 import _lib as L
from sres_b200 import nn as _snn
from sres_b200.parallel import dp_schedule, gather_rows, shard_range

TensorOrTensors = Union[Tensor, Sequence[Tensor]]


def ttsplit_times(times: List[int]) -> Dict[TSet, List[int]]:
    """dual_trainer.py:28-36."""
    start, result, nt = 0, {}, len(times)
    for tset, frac in cfg().task.ttsplit.items():
        end = start + int(frac * nt)
        result[TSet(tset)] = times[start:end]
        start = end
    return result


def denorm(t: Tensor, norm_data: Dict[str, Any]) -> Tensor:
    """dual_trainer.py:67-77, kept on the device (x*std+mean, then optional min/max rescale)."""
    normed = t.detach()
    if "mean" in norm_data:
        normed = (normed * norm_data["std"]) + norm_data["mean"]
    if "max" in norm_data:
        normed = (normed * (norm_data["max"] - norm_data["min"])) + norm_data["min"]
    return normed


class ModelTrainer(object):

    def __init__(self, cc: ConfigContext, dataset: Optional[BatchDataset] = None):
        self.device: torch.device = set_device()
        self.model_manager: SRModels = SRModels(self.device)
        if dataset is not None:
            self.model_manager._dataset = dataset
        self.context = cc
        self.min_loss = float("inf")
        self.eps = 1e-6
        self.scheduler = None
        self.model = self.model_manager.get_model()
        lr, wd = cfg().task.lr, cfg().task.get("weight_decay", 0.0)
        if cfg().pipeline.get("fused_adam", True):
            self.optimizer = _snn.FusedAdam(self.model, lr=lr, weight_decay=wd)
        else:  # the reference's optimizer works too: parameters are ordinary nn.Parameters
            self.optimizer = torch.optim.Adam(self.model.parameters(), lr=lr, weight_decay=wd)
        self.checkpoint_manager = CheckpointManager(self.model, self.optimizer)
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        if self.world > 1:
            self.model.enable_data_parallel()
            # every rank starts from rank 0's weights (constructors draw from per-process RNG state)
            dist.broadcast(self.model.engine.flat, src=0)
            self.model.engine.mark_params_changed()
        self.input, self.target, self.product, self.interp = {}, {}, {}, {}
        self.current_losses: Dict[str, float] = {}
        self.time_index: int = -1
        self.tile_index: int = -1
        self.validation_loss: float = float("inf")
        self.data_timestamps: Dict[TSet, List[int]] = {}
        self.eval_history: Dict[TSet, List[Dict[str, float]]] = {}
        self.train_state = None

    # -- plumbing ----------------------------------------------------------------------------------
    def _sync_python_rng(self):
        """Data parallel only: the timeslice order, the tile-batch shuffle and the flip index are drawn from Python's
        `random` (like the reference); all ranks must draw the same ones or they would walk different timeslices and
        issue different numbers of collectives.  Rank 0's next draw seeds everybody."""
        if self.world > 1:
            s = torch.tensor([random.getrandbits(62)], dtype=torch.int64, device=self.device)
            dist.broadcast(s, src=0)
            random.seed(int(s.item()))

    def get_dataset(self) -> BatchDataset:
        return self.model_manager.get_dataset()

    @property
    def target_variables(self) -> List[str]:
        return list(cfg().task.target_variables)

    def load_timeslice(self, ctime, **kwargs) -> Optional[TileArray]:
        return self.get_dataset().load_timeslice(ctime, **kwargs)

    def get_srbatch(self, ctile: Dict[str, int], ctime, **kwargs) -> Optional[TileArray]:
        return self.get_dataset().get_batch_array(ctile, ctime, **kwargs)

    def init_data_timestamps(self):
        if len(self.data_timestamps) == 0:
            ctimes = self.get_dataset().get_dset_time_indices()
            random.shuffle(ctimes)
            self.data_timestamps = ttsplit_times(ctimes)

    # -- the hot path ------------------------------------------------------------------------------
    def apply_network(self, target_data) -> Tuple[Tensor, TensorOrTensors, Tensor]:
        """(input, product, target) of one HR batch: bicubic down + model (dual_trainer.py:557-571).
        Errors propagate (the reference swallows them and returns None, logging.py:13-20)."""
        data = target_data.data if isinstance(target_data, TileArray) else target_data
        input_tensor: Tensor = array2tensor(data)
        dsample = cfg().task.get("data_downsample", 1.0)
        if dsample > 1.0:
            input_tensor = downsample(input_tensor, scale_factor=dsample)
        target_channels: List[str] = self.target_variables
        output_tensor: Tensor = input_tensor
        if input_tensor.shape[1] > len(target_channels):
            tindx = torch.tensor(self.get_dataset().get_channel_idxs(target_channels), device=input_tensor.device)
            output_tensor = torch.index_select(input_tensor, 1, tindx)
        input_tensor = downsample(input_tensor)
        result_tensor: TensorOrTensors = self.model(input_tensor)
        return input_tensor, result_tensor, output_tensor

    def charbonnier(self, prd: Tensor, tar: Tensor) -> Tensor:
        return _snn.loss(prd, tar, "charbonnier", self._loss_group())

    def _loss_group(self):
        return dist.group.WORLD if (self.world > 1 and self.model.training and torch.is_grad_enabled()) else None

    def conform_to_product(self, prd: Tensor, tar: Tensor) -> Tensor:
        return tar  # the CUDA loss crops the target to the product's (H,W) itself (dual_trainer.py:200-203)

    def single_product_loss(self, prd: Tensor, tar: Tensor, weight: float = 1.0) -> Tensor:
        fn = cfg().model.loss_fn
        if fn not in ("l2", "charbonnier", "l1"):
            raise Exception("Unknown single-product loss function {}".format(fn))
        return _snn.loss(prd, tar, fn, self._loss_group(), weight)

    def loss(self, products: TensorOrTensors, target: Tensor, weight: float = 1.0) -> Tuple[float, Tensor]:
        """(python float, differentiable tensor) like dual_trainer.py:221-234 (`.item()` syncs)."""
        if isinstance(products, torch.Tensor):
            sloss = self.single_product_loss(products, target, weight)
            return sloss.item(), sloss
        raise NotImplementedError("multi-scale product lists are not produced by RCAN")

    def train_step(self, batch) -> Tensor:
        """One optimizer step on one HR tile batch: zero_grad, forward, loss, backward, step
        (dual_trainer.py:310-323 without the logging).  Returns the loss as a device scalar."""
        self.optimizer.zero_grad()
        _, boutput, btarget = self.apply_network(batch)
        mloss = self.single_product_loss(boutput, btarget)
        mloss.backward()
        self.optimizer.step()
        return mloss.detach()

    def train_stream(self, host_batches):
        """Optimizer steps over an iterable of HOST batches (pinned memory for a truly asynchronous copy): the host-to-device
        copy of batch i+1 is issued on a copy stream before step i is enqueued, so it runs under step i's kernels instead of
        in front of step i+1's.  Yields each step's loss as a device scalar (reading it with .item() does not wait for the
        next batch's copy).  Same arithmetic as calling train_step batch by batch."""
        dev = self.device
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)

        def stage(hb):
            data = hb.data if isinstance(hb, TileArray) else hb
            if not isinstance(data, torch.Tensor):
                data = torch.from_numpy(np.ascontiguousarray(data))
            with torch.cuda.stream(self._copy_stream):
                d = data.to(device=dev, dtype=torch.float32, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            d.record_stream(main)          # allocated on the copy stream, consumed on the compute stream
            return d, ev

        it = iter(host_batches)
        try:
            nxt = stage(next(it))
        except StopIteration:
            return
        while nxt is not None:
            cur, ev = nxt
            try:
                nxt = stage(next(it))
            except StopIteration:
                nxt = None
            main.wait_event(ev)
            yield self.train_step(cur)

    # -- training loop -----------------------------------------------------------------------------
    def train(self, nepochs: int, refresh_state: bool, **kwargs) -> Dict[str, float]:
        if nepochs == 0:
            return {}
        interp_loss = kwargs.get("interp_loss", False)
        seed = kwargs.get("seed", 4456)
        verbose = kwargs.get("verbose", True)
        torch.manual_seed(seed)
        torch.cuda.manual_seed(seed)
        self.scheduler = kwargs.get("scheduler", None)
        epoch0, itime0, epoch_loss, interp_sloss, tset = 1, 0, 0.0, 0.0, TSet.Train
        train_start = time.time()
        if refresh_state:
            if self.rank == 0:
                self.checkpoint_manager.clear_checkpoints()
        else:
            self.train_state = self.checkpoint_manager.load_checkpoint(TSet.Train, update_model=True)
            epoch0 = self.train_state.get("epoch", 1)
            itime0 = self.train_state.get("itime", 0)
            epoch_loss = self.train_state.get("loss", float("inf"))
            nepochs += epoch0
        self._sync_python_rng()
        self.init_data_timestamps()
        for epoch in range(epoch0, nepochs):
            self.model.train()
            nts = len(self.data_timestamps[TSet.Train])
            for itime in range(itime0, nts):
                ctime = self.data_timestamps[TSet.Train][itime]
                timeslice = self.load_timeslice(ctime)
                tile_iter = TileIterator.get_iterator(ntiles=timeslice.sizes["tiles"], randomize=True)
                binput = boutput = btarget = None
                batches = list(iter(tile_iter))
                # data parallel: every global step consumes `world` consecutive batches of the shuffled order; in a ragged
                # last step the ranks without a batch re-run one with loss weight 0 (sres_b200.parallel.dp_schedule)
                for ibatch, weight in dp_schedule(len(batches), self.rank, self.world):
                    ctile = batches[ibatch]
                    batch_data = self.get_srbatch(ctile, ctime)
                    if batch_data is None:
                        break
                    self.optimizer.zero_grad()
                    binput, boutput, btarget = self.apply_network(batch_data)
                    [sloss, mloss] = self.loss(boutput, btarget, weight)
                    tile_iter.register_loss("model", sloss)
                    if interp_loss:
                        with torch.no_grad():
                            [interp_sloss, _] = self.loss(upsample(binput), btarget)
                        tile_iter.register_loss("interpolated", interp_sloss)
                    if verbose and self.rank == 0:
                        pct = (sloss / interp_sloss) * 100 if interp_sloss else float("nan")
                        print(f" ** <{self.model_manager.model_name}> TRAIN E({epoch:3}/{nepochs}) TIME[{itime:3}:{ctime:4}] "
                              f"TILES[{ctile['start']:4}:{ctile['end']:4}][F{batch_data.attrs.get('xyflip', 0)}]-> "
                              f"Loss= {sloss*1000:6.2f} ({interp_sloss*1000:6.2f}): {pct:.2f}%", flush=True)
                    mloss.backward()
                    self.optimizer.step()
                if binput is not None:
                    self.input[tset] = binput.detach().cpu().numpy()
                    self.target[tset] = btarget.detach().cpu().numpy()
                    self.product[tset] = boutput.detach().cpu().numpy()
                epoch_loss = tile_iter.accumulate_loss("model") if tile_iter.batch_losses("model") else epoch_loss
                il = tile_iter.accumulate_loss("interpolated") if tile_iter.batch_losses("interpolated") else 0.0
                if self.rank == 0 and cfg().task.get("checkpoint_every_timeslice", True):
                    self.checkpoint_manager.save_checkpoint(epoch, itime, TSet.Train, epoch_loss, il)
            if self.scheduler is not None:
                self.scheduler.step()
            # epoch-end validation pass; a new best model loss writes the validation checkpoint (dual_trainer.py:333-338, 534-539)
            self.record_eval(epoch, {TSet.Train: epoch_loss}, TSet.Validation)
            self.model.train()
            itime0 = 0
        train_time = time.time() - train_start
        ntotal_params = sum(p.numel() for p in self.model.parameters() if p.requires_grad)
        self.record_eval(nepochs, {}, TSet.Test)
        if self.rank == 0:
            print(f" -------> Training model with {ntotal_params} wts took {train_time/60:.2f} min.")
        self.current_losses = dict(prediction=epoch_loss)
        return self.current_losses

    # -- inference ---------------------------------------------------------------------------------
    def process_image(self, tset: TSet, itime: int, **kwargs):
        """Tile -> batched forward -> stitch for one timeslice (dual_trainer.py:396-447).  Returns
        (images[var][type] -> 2-D numpy array, losses[var] -> dict(model, interpolated))."""
        seed = kwargs.get("seed", 333)
        cfg().task["xyflip"] = False
        torch.manual_seed(seed)
        if kwargs.get("update_model", False):
            self.train_state = self.checkpoint_manager.load_checkpoint(TSet.Validation, **kwargs)
        self.time_index = itime
        self._sync_python_rng()
        self.init_data_timestamps()
        ctime = kwargs.get("ctime", None)
        if ctime is None:
            ctime = self.data_timestamps[TSet.Train][itime]
        timeslice = self.load_timeslice(ctime)
        vnames, cvar = self.target_variables, kwargs.get("var", None)
        output_vars = [cvar] if cvar is not None else vnames
        model_losses, interp_losses, batches, stats = [], [], [], []
        tile_iter = TileIterator.get_iterator(ntiles=timeslice.sizes["tiles"])
        ctiles = list(iter(tile_iter))
        # data parallel: rank r runs the forward on a contiguous range of the tile batches; the products are gathered
        # so every rank (rank 0 in practice) can stitch the full image (SURVEY.md 8e)
        lo, hi = shard_range(len(ctiles), self.rank, self.world) if self.world > 1 else (0, len(ctiles))
        with torch.no_grad():
            for ctile in ctiles[lo:hi]:
                batch_data = self.get_srbatch(ctile, ctime, shuffle=False)
                if batch_data is None:
                    break
                binput, boutput, btarget = self.apply_network(batch_data)
                binterp = upsample(binput)
                # the per-batch losses stay on the device: one host sync per image, not two per batch
                model_losses.append(self.single_product_loss(boutput, btarget))
                interp_losses.append(self.single_product_loss(binterp, btarget))
                # products stay normalised; x*std+mean (dual_trainer.py:67-77) is fused into the stitch kernel
                batches.append(dict(input=binput, target=btarget, interpolated=binterp, model=boutput))
                stats.append(batch_data.attrs)
        nb = len(model_losses)
        lsum = torch.stack([torch.stack(model_losses).double().sum(), torch.stack(interp_losses).double().sum(),
                            torch.tensor(float(nb), dtype=torch.float64, device=self.device)]) if nb else \
            torch.zeros(3, dtype=torch.float64, device=self.device)
        if self.world > 1:
            ntiles = int(timeslice.sizes["tiles"])
            counts = []   # tile rows per rank (equal batch sizes except the last batch)
            for r in range(self.world):
                rlo, rhi = shard_range(len(ctiles), r, self.world)
                counts.append(sum(min(c["end"], ntiles) - c["start"] for c in ctiles[rlo:rhi]))
            nch, hr_y, hr_x = len(self.target_variables), int(timeslice.shape[2]), int(timeslice.shape[3])
            dsample = int(cfg().task.get("data_downsample", 1.0))
            scale = int(np.prod(cfg().model.downscale_factors)) * dsample
            merged = {}
            for k in ("input", "target", "interpolated", "model"):
                f = scale if k == "input" else dsample
                local = torch.cat([denorm(bd[k], a).float() for bd, a in zip(batches, stats)], dim=0) if batches else None
                merged[k] = gather_rows(local, counts, (nch, hr_y // f, hr_x // f), self.device)
            batches, stats = [merged], None
            dist.all_reduce(lsum)
        lsum = lsum.cpu()
        mean_model = float(lsum[0] / lsum[2]) if float(lsum[2]) > 0 else float("nan")
        mean_interp = float(lsum[1] / lsum[2]) if float(lsum[2]) > 0 else float("nan")
        images, losses = {}, {}
        # data parallel: the stitched images are built (and copied to the host) on rank 0 only -- eight ranks each pulling
        # 2.4 GB of float64 images through the same host memory made the 8-GPU pass slower than one GPU (all_ranks=True
        # restores the replicated result)
        stitch_here = self.world == 1 or self.rank == 0 or kwargs.get("all_ranks", False)
        for ivar, vname in enumerate(output_vars):
            if stitch_here:
                images[vname] = self.assemble_images(batches, ivar, timeslice.coords["tiles"], timeslice.attrs["grid_shape"], stats)
            losses[vname] = dict(model=mean_model, interpolated=mean_interp)
        return images, losses

    def assemble_images(self, batches: List[Dict[str, Tensor]], ivar: int, tile_ids, grid_shape: Dict[str, int],
                        norm_stats: Optional[List[Dict[str, Any]]] = None) -> Dict[str, np.ndarray]:
        """Place tile `tid` at grid cell (tid // gx, tid % gx), NaN elsewhere (dual_trainer.py:449-480), on the GPU.
        norm_stats (one dict(mean, std) of shape (B,C,1,1) per batch): the tiles are normalised and the kernel
        de-normalises them, x*std+mean, while it places them (`denorm`, dual_trainer.py:67-77, same two fp32 roundings).
        dtype rule of the reference's np.block: float64 iff at least one cell stayed empty (its placeholder is a
        float64 NaN tile); the widening runs on the device and every image reaches the host through ONE copy into
        pinned memory (torch's caching host allocator recycles the buffers of images the caller has dropped)."""
        lib = L.lib()
        gy, gx = int(grid_shape["y"]), int(grid_shape["x"])
        tile_ids = np.asarray(tile_ids)
        mean = std = None
        if norm_stats is not None:
            if any("max" in a for a in norm_stats):
                raise NotImplementedError("sres (B200 build): min/max de-normalisation has no CUDA kernel (lnorm only)")
            mean = torch.cat([torch.as_tensor(a["mean"], device=self.device).float().reshape(-1) for a in norm_stats]).contiguous()
            std = torch.cat([torch.as_tensor(a["std"], device=self.device).float().reshape(-1) for a in norm_stats]).contiguous()
        pending: Dict[str, Tensor] = {}
        for image_type in batches[0].keys():
            tiles = torch.cat([torch.as_tensor(b[image_type], device=self.device).detach().float() for b in batches], dim=0).contiguous()
            n, Cc, th, tw = tiles.shape
            cell = np.full(gy * gx, -1, dtype=np.int32)
            cell[tile_ids[:n].astype(np.int64)] = np.arange(n, dtype=np.int32)   # (ids are unique: later == earlier)
            cell_d = torch.from_numpy(cell).to(self.device)
            img = torch.empty(gy * th, gx * tw, dtype=torch.float32, device=self.device)
            if mean is not None and mean.numel() != n * Cc:
                raise ValueError(f"assemble_images: {mean.numel()} normalisation entries for {n} tiles x {Cc} channels")
            L.check(lib.sres_tiles_stitch_hw(L.ptr(tiles), Cc, ivar, th, tw, gy, gx, L.ptr(cell_d), L.ptr(mean), L.ptr(std),
                                             L.ptr(img), L.cur_stream()), "sres_tiles_stitch_hw")
            dev_img = img.double() if (cell < 0).any() else img
            host = torch.empty(dev_img.shape, dtype=dev_img.dtype, pin_memory=True)
            host.copy_(dev_img, non_blocking=True)
            pending[image_type] = host
        torch.cuda.current_stream().synchronize()
        return {k: v.numpy() for k, v in pending.items()}

    def record_eval(self, epoch: int, losses: Dict[TSet, float], tset: TSet, **kwargs) -> Optional[Dict[str, float]]:
        """Evaluate `tset` when the train/test split gives it any timeslices and log the result (dual_trainer.py:349-358;
        the reference's CSV results accumulator is outside the hot path: the history is kept in memory)."""
        if cfg().task.ttsplit.get(tset.value, 0.0) <= 0.0:
            return None
        self.init_data_timestamps()
        if not self.data_timestamps.get(tset):
            return None
        saved_ti = self.time_index
        self.time_index = -1            # every timeslice of the set
        try:
            _, eval_losses = self.evaluate(tset, update_model=False, epoch=epoch, keep_results=False, **kwargs)
        finally:
            self.time_index = saved_ti
        self.eval_history.setdefault(tset, []).append(dict(epoch=epoch, **eval_losses, **{f"{k.value}_loss": v for k, v in losses.items()}))
        if self.rank == 0 and kwargs.get("verbose", False):
            print(f" --->> record {tset.name} eval[{epoch}]: eval_losses={eval_losses}, losses={losses}")
        return eval_losses

    def evaluate(self, tset: TSet, **kwargs):
        """Batched forward over the tiles of the validation / test timeslices (dual_trainer.py:482-543).
        Returns (dict(input,target,model,interpolated) -> numpy (N,C,·,·), dict(model, interpolated)).  For the validation
        set a model loss below the best one so far writes the validation checkpoint (:534-539); the best-so-far comes
        from that checkpoint's `loss` entry (update_checkpoint, default on), the model itself is only reloaded when
        update_model is passed."""
        assert tset in [TSet.Validation, TSet.Test], f"Invalid tset in training evaluation: {tset.name}"
        self.time_index = kwargs.get("time_index", self.time_index)
        epoch = kwargs.get("epoch", None)
        update_checkpoint = kwargs.get("update_checkpoint", True)
        if update_checkpoint:
            state = self.checkpoint_manager.load_checkpoint(TSet.Validation, update_model=kwargs.get("update_model", False), quiet=True)
            self.validation_loss = state.get("loss", float("inf"))
            if epoch is None:
                epoch = state.get("epoch", 0)
        self._sync_python_rng()
        self.init_data_timestamps()
        ml, il, res = [], [], dict(input=[], target=[], model=[], interpolated=[])
        with torch.no_grad():
            for itime, ctime in enumerate(self.data_timestamps.get(tset, [])):
                if (self.time_index < 0) or (itime == self.time_index):
                    timeslice = self.load_timeslice(ctime)
                    for ctile in iter(TileIterator.get_iterator(ntiles=timeslice.sizes["tiles"])):
                        batch_data = self.get_srbatch(ctile, ctime)
                        if batch_data is None:
                            break
                        binput, boutput, btarget = self.apply_network(batch_data)
                        binterp = upsample(binput)
                        ml.append(self.loss(boutput, btarget)[0])
                        il.append(self.loss(binterp, btarget)[0])
                        if kwargs.get("keep_results", True):
                            for k, v in zip(res.keys(), (binput, btarget, boutput, binterp)):
                                res[k].append(v.detach())
                    if self.time_index >= 0:
                        break
        shapes = sorted({tuple(v.shape[2:]) for v in res["target"]})
        if len(shapes) > 1:
            # the reference's np.concatenate fails on the same batches
            raise ValueError(f"evaluate(keep_results=True): the batches come in tile shapes {shapes} (rectangular tiles with "
                             "task.xyflip transpose some of them) and cannot be concatenated; use keep_results=False or "
                             "turn xyflip off")
        results = {k: (torch.cat(v).cpu().numpy() if v else None) for k, v in res.items()}
        losses = dict(model=float(np.mean(ml)) if ml else float("nan"), interpolated=float(np.mean(il)) if il else float("nan"))
        if tset == TSet.Validation and ml and self.time_index < 0:
            if losses["model"] < self.validation_loss or self.validation_loss == 0.0:
                if update_checkpoint and self.validation_loss > 0.0 and self.rank == 0:
                    self.checkpoint_manager.save_checkpoint(epoch or 0, 0, TSet.Validation, losses["model"], losses["interpolated"])
                self.validation_loss = losses["model"]
        return results, losses
