"""Tensor / interpolation helpers, mirror of sres/base/util/array.py:37-41, 67-76, 84-87."""
import math
from typing import Union

import numpy as np
import torch

from sres.base.gpu import get_device
from sres.base.util.config import cfg
from sres_b200 import nn as _snn
from sres_b200._lib import RESIZE_MODES

Tensor = torch.Tensor


def torch_interp_mode(downsample: bool) -> str:
    mode = cfg().task.downsample_mode if downsample else cfg().task.upsample_mode
    if mode == "linear":
        return "bilinear"
    if mode == "cubic":
        return "bicubic"
    return mode


def _values(darray) -> np.ndarray:
    return darray.values if hasattr(darray, "values") and not isinstance(darray, np.ndarray) else darray


def array2tensor(darray) -> Tensor:
    """fp32 tensor on the device with requires_grad=True (array.py:67-70).  Device tensors pass through."""
    if isinstance(darray, torch.Tensor):
        return darray.detach().to(device=get_device(), dtype=torch.float32, non_blocking=True).requires_grad_(True)
    nparray = np.ascontiguousarray(_values(darray))
    return torch.tensor(nparray, device=get_device(), requires_grad=True, dtype=torch.float32)


def _resize(t: Tensor, factor: float, down: bool) -> Tensor:
    mode = torch_interp_mode(down)
    if mode == "bicubic":
        return _snn.bicubic_resize(t, factor)
    if mode not in RESIZE_MODES:
        raise ValueError(f"sres (B200 build): interpolation mode '{mode}' is not supported; task.downsample_mode / "
                         "upsample_mode accepts cubic, linear, nearest, nearest-exact, area (or bicubic, bilinear)")
    return _snn.resize(t, factor, mode)


def downsample(target_data, **kwargs) -> Tensor:
    scale_factor = kwargs.get("scale_factor", math.prod(cfg().model.downscale_factors))
    t = target_data if isinstance(target_data, torch.Tensor) else array2tensor(target_data)
    return _resize(t, 1.0 / scale_factor, True)


def upsample(input_tensor: Tensor) -> Tensor:
    return _resize(input_tensor, math.prod(cfg().model.downscale_factors), False)
