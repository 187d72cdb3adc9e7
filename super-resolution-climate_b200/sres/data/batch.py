"""Device-resident tile batches: the loader side of the hot path.

Mirrors, for the tile path only:
  SWOTRawDataLoader.load_timeslice / get_tiles   sres/base/source/swot/raw.py:147-153, 216-233
  SWOTRawDataLoader.select_batch / norm('lnorm') sres/base/source/swot/raw.py:160-183, 211-214
  xyflip                                         sres/base/source/batch.py:33-49
  BatchDataset.load_timeslice / get_batch_array  sres/data/batch.py:137-142
The reference reads LLC4320 binary files (out of scope here: there is no data in the box); the
region source is pluggable: `dataset.source: synthetic` (seeded field with NaN land patches) or a
user-supplied callable returning the (C,Y,X) float32 region of a time index.  Everything after the
region is on the GPU: tile extraction, NaN-tile drop, per-tile normalisation and the flip.
"""
import ctypes as C
import random
from typing import Callable, Dict, List, Optional

import numpy as np
import torch

from sres.base.gpu import get_device
from sres.base.util.config import cfg
from sres.data.tiles import TileGrid
from sres_b200 import _lib as L


class TileArray:
    """Just enough of xarray.DataArray for the trainer: data on the device, named dims, coords, attrs."""

    def __init__(self, data: torch.Tensor, dims, coords=None, attrs=None):
        self.data, self.dims = data, tuple(dims)
        self.coords, self.attrs = dict(coords or {}), dict(attrs or {})

    @property
    def shape(self):
        return tuple(self.data.shape)

    @property
    def sizes(self) -> Dict[str, int]:
        return dict(zip(self.dims, self.data.shape))

    @property
    def values(self) -> np.ndarray:
        return self.data.detach().cpu().numpy()

    def mean(self):
        return float(torch.nanmean(self.data))

    def std(self):
        return float(self.data[torch.isfinite(self.data)].std())


def synthetic_region(C_: int, Y: int, X: int, seed: int, nan_fraction: float = 0.2) -> np.ndarray:
    """Seeded smooth field + noise with rectangular NaN 'land' patches shared by all variables."""
    rng = np.random.default_rng(seed)
    yy, xx = np.meshgrid(np.arange(Y, dtype=np.float32), np.arange(X, dtype=np.float32), indexing="ij")
    out = np.empty((C_, Y, X), dtype=np.float32)
    for c in range(C_):
        out[c] = np.sin(xx / 37.0 + c) * np.cos(yy / 29.0) * (3.0 + c) + 20.0 * (c + 1)
        out[c] += rng.standard_normal((Y, X), dtype=np.float32) * 0.1
    npatch = max(1, int(nan_fraction * (Y // 192) * (X // 192) / 2))
    for _ in range(npatch):
        y0, x0 = int(rng.integers(0, Y)), int(rng.integers(0, X))
        out[:, y0:y0 + int(rng.integers(8, 260)), x0:x0 + int(rng.integers(8, 260))] = np.nan
    return out


def source_table(flags: np.ndarray, C_: int, ncand: int, order: str):
    """Which candidate tile feeds slot (n, c) of the (N,C,Th,Tw) result, and the tile-id coordinate.

    order == 'reference': bit-exact restatement of raw.py:225-233 -- survivors of the channel-major
    flat list are re-chunked C at a time (so for C > 1 a slot pairs consecutive flat tiles, SURVEY.md 8a)
    and the reshape raises when the survivor count is not a multiple of C.
    order == 'corrected': slot (n, c) is tile n of variable c; a tile is dropped when any variable is
    non-finite there."""
    if order == "reference":
        surv = np.nonzero(flags)[0]
        if surv.size % C_ != 0:
            raise ValueError(f"cannot reshape array of size {surv.size} tiles into shape ({surv.size // C_},{C_},...)")
        n = surv.size // C_
        return surv.astype(np.int32), surv[:n].astype(np.int64)
    if order == "corrected":
        ok = flags.reshape(C_, ncand).all(axis=0)
        ids = np.nonzero(ok)[0]
        src = (np.arange(C_)[None, :] * ncand + ids[:, None]).reshape(-1)
        return src.astype(np.int32), ids.astype(np.int64)
    raise ValueError(f"tile_order must be 'reference' or 'corrected', got {order!r}")


class BatchDataset(object):

    def __init__(self, task_config=None, region_source: Optional[Callable[[int], np.ndarray]] = None):
        self.task = task_config if task_config is not None else cfg().task
        self.varnames: List[str] = list(self.task.input_variables.keys())
        self.tile_grid = TileGrid()
        self.region_source = region_source
        self.time_index = -1
        self.timeslice: Optional[TileArray] = None
        self.lib = L.lib()

    # -- regions ---------------------------------------------------------------------------------
    def _llc_reader(self):
        """`dataset.source: llc4320`: the raw LLC4320 files of config/dataset/swot_*.yaml (sres/data/llc4320.py)."""
        if getattr(self, "_llc", None) is None:
            from sres.data.llc4320 import LLC4320Reader
            ds = cfg().dataset
            self._llc = LLC4320Reader(str(ds.dataset_root), str(ds.dataset_files), str(ds.template), ds.get("roi", None),
                                      int(ds.get("nx", 4320)), get_device())
        return self._llc

    def get_dset_time_indices(self) -> List[int]:
        if self.region_source is None and cfg().dataset.get("source", "synthetic") == "llc4320":
            return self._llc_reader().time_indices(self.varnames[0])
        return list(range(int(cfg().dataset.get("ntimes", 1))))

    def load_region_data(self, time_index: int, **kwargs):
        """(C,Y,X) float32 region of a time index: a host array, or a device tensor when the source already lives there."""
        if self.region_source is not None:
            reg = self.region_source(time_index)
            return reg if isinstance(reg, torch.Tensor) else np.ascontiguousarray(reg, dtype=np.float32)
        ds = cfg().dataset
        if ds.get("source", "synthetic") == "llc4320":
            return self._llc_reader().load_region_data(self.varnames, time_index)
        if ds.get("source", "synthetic") != "synthetic":
            raise NotImplementedError(f"sres (B200 build): dataset.source '{ds.get('source')}' -- use synthetic, llc4320 or a "
                                      "region_source callable")
        return synthetic_region(len(self.varnames), int(ds.region["ys"]), int(ds.region["xs"]),
                                int(ds.get("seed", 0)) + 1000 * int(time_index), float(ds.get("nan_fraction", 0.2)))

    # -- tiles -----------------------------------------------------------------------------------
    def get_tiles(self, region: torch.Tensor) -> TileArray:
        """(C,Y,X) device region -> TileArray(tiles, channels, y, x), raw.py:216-233 on the GPU."""
        C_, Y, X = region.shape
        ts = self.tile_grid.get_full_tile_size()
        Th, Tw = ts["y"], ts["x"]
        gs = self.tile_grid.get_grid_shape(image_shape=dict(c=C_, y=Y, x=X))
        roi = self.tile_grid.get_active_region(image_shape=dict(c=C_, y=Y, x=X))
        gy, gx, y0, x0 = gs["y"], gs["x"], roi["y"][0], roi["x"][0]
        ncand = gy * gx
        dev = region.device
        flags = torch.empty(C_ * ncand, dtype=torch.int32, device=dev)
        st = L.cur_stream()
        L.check(self.lib.sres_tiles_finite_flags_hw(L.ptr(region), C_, Y, X, y0, x0, Th, Tw, gy, gx, L.ptr(flags), st),
                "sres_tiles_finite_flags_hw")
        src, ids = source_table(flags.cpu().numpy(), C_, ncand, self.task.get("tile_order", "reference"))
        n = src.size // C_
        out = torch.empty(n, C_, Th, Tw, dtype=torch.float32, device=dev)
        if n > 0:
            src_d = torch.from_numpy(src).to(dev)
            L.check(self.lib.sres_tiles_gather_hw(L.ptr(region), C_, Y, X, y0, x0, Th, Tw, gy, gx, L.ptr(src_d), n * C_,
                                                  L.ptr(out), st), "sres_tiles_gather_hw")
        return TileArray(out, ["tiles", "channels", "y", "x"], coords=dict(tiles=ids, channels=self.varnames),
                         attrs=dict(grid_shape=dict(gs)))

    def load_timeslice(self, time_index: int, **kwargs) -> TileArray:
        if time_index != self.time_index:
            region = self._load_region_on_device(time_index)
            self.timeslice = self.get_tiles(region)
            self.time_index = time_index
        return self.timeslice

    def _load_region_on_device(self, time_index: int) -> torch.Tensor:
        """The (C,Y,X) region of a time index on this rank's GPU.  Under torch.distributed every rank needs the same region
        (tile ids are global): rank 0 reads / generates it, copies it to its GPU once and broadcasts it over NVLink, instead
        of every rank pulling the same hundreds of megabytes through host memory."""
        import torch.distributed as dist
        dev = get_device()
        world = dist.get_world_size() if dist.is_initialized() else 1
        if world == 1 or dev.type != "cuda":
            region = self.load_region_data(time_index)
            region = (region if isinstance(region, torch.Tensor) else torch.from_numpy(region)).to(dev, non_blocking=True)
            return region.contiguous().float()
        if dist.get_rank() == 0:
            region = self.load_region_data(time_index)
            region = (region if isinstance(region, torch.Tensor) else torch.from_numpy(region)).to(dev, non_blocking=True).contiguous().float()
            shape = torch.tensor(list(region.shape), dtype=torch.int64, device=dev)
        else:
            region, shape = None, torch.zeros(3, dtype=torch.int64, device=dev)
        dist.broadcast(shape, src=0)
        if region is None:
            region = torch.empty(tuple(int(v) for v in shape.tolist()), dtype=torch.float32, device=dev)
        dist.broadcast(region, src=0)
        return region

    # -- batches ---------------------------------------------------------------------------------
    def select_batch(self, tile_range) -> Optional[TileArray]:
        """raw.py:160-167 + norm: slice [start, min(end, N)), normalise (and flip) on the device."""
        ts = self.timeslice
        ntiles = ts.shape[0]
        if tile_range[0] < ntiles:
            end = min(tile_range[1], ntiles)
            raw = ts.data[tile_range[0]:end]
            return self.norm(raw, (tile_range[0], end))
        return None

    def norm(self, raw: torch.Tensor, tile_range, flip_index: int = 0) -> TileArray:
        ntype = self.task.norm
        if ntype != "lnorm":
            raise NotImplementedError(f"sres (B200 build): norm '{ntype}' has no CUDA kernel (lnorm only)")
        B, C_, Th, Tw = raw.shape
        raw = raw.contiguous()
        # flips 4-7 end with swapaxes(-1, -2) (source/batch.py:37-49): a (Th, Tw) tile comes out (Tw, Th)
        out = torch.empty((B, C_, Tw, Th) if int(flip_index) & 4 else (B, C_, Th, Tw), dtype=raw.dtype, device=raw.device)
        mean = torch.empty(B, C_, 1, 1, dtype=torch.float32, device=raw.device)
        std = torch.empty_like(mean)
        L.check(self.lib.sres_tiles_lnorm_hw(L.ptr(raw), B * C_, Th, Tw, int(flip_index), L.ptr(out), L.ptr(mean), L.ptr(std),
                                             L.cur_stream()), "sres_tiles_lnorm_hw")
        return TileArray(out, ["tiles", "channels", "y", "x"],
                         coords=dict(tiles=self.timeslice.coords["tiles"][tile_range[0]:tile_range[1]], channels=self.varnames),
                         attrs=dict(mean=mean, std=std, xyflip=int(flip_index)))

    def get_batch_array(self, ctile: Dict[str, int], ctime: int, **kwargs) -> Optional[TileArray]:
        """BatchDataset.get_batch_array (data/batch.py:137-142): select, normalise, xyflip.  The flip
        index comes from Python's `random.randint(0, 7)` exactly like source/batch.py:40."""
        self.load_timeslice(ctime)
        ts = self.timeslice
        if ctile["start"] >= ts.shape[0]:
            return None
        end = min(ctile["end"], ts.shape[0])
        flip = random.randint(0, 7) if self.task.get("xyflip", False) else 0
        return self.norm(ts.data[ctile["start"]:end], (ctile["start"], end), flip)

    def get_channel_idxs(self, channels: List[str]) -> List[int]:
        return [self.varnames.index(c) for c in channels]
