"""Nearest, nearest-exact, bilinear and area resize (`sres_resize`, `sres_b200.nn.resize`) and the task settings that
select them (`task.downsample_mode` / `task.upsample_mode`, sres/base/util/array.py:37-41, 72-76, 84-87).

Checked here:

  * without a GPU: `sres_resize` refuses null pointers, bad shapes, unknown modes and bad scales before it touches
    anything; `torch_interp_mode` maps the config names; `_resize` refuses a mode it has no kernel for with ValueError;
  * kernel by kernel against F.interpolate on the same input: every mode, down and up, factors 2, 3, 4 and 8, square and
    non-square planes, sizes the factor does not divide, 1 to 64 * 16 planes, outputs pre-filled with NaN and followed by
    a guard region.  nearest / nearest-exact are bit-identical to torch's CPU and CUDA results; bilinear and area are
    within 1e-6 of the CPU result relative to F.interpolate(|x|), the sum of the weighted magnitudes (both modes have
    non-negative weights);
  * the controller end to end with non-bicubic modes: the network input `apply_network` builds (with and without the
    `data_downsample` pre-step), training steps, and the "interpolated" product of `process_image` and `evaluate`.
"""
import ctypes as C
import math
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

NEW_MODES = ["nearest", "nearest-exact", "bilinear", "area"]
FACTORS = [2, 3, 4, 8]
REL = 1e-6
GUARD, SENTINEL = 64, 12345.0


@pytest.fixture(scope="module")
def lib():
    from sres_b200 import _lib as L
    lb = L.lib()
    lb.sres_last_error.restype = C.c_char_p
    return lb


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_header_declares_resize_and_its_modes():
    import os
    from sres_b200 import _lib as L
    text = open(os.path.join(os.path.dirname(__file__), "..", "include", "sres_b200.h")).read()
    assert "SRES_API int sres_resize(" in text
    for name, code in L.RESIZE_MODES.items():
        assert f"#define SRES_RESIZE_{name.upper().replace('-', '_')} {code}" in text


def test_resize_rejects_bad_arguments(lib):
    """Fake device pointers: every call below must be refused before anything is dereferenced or enqueued."""
    p = C.c_void_p(16)
    good = (p, p, 2, 8, 8, 4, 4, 2.0, 2.0)

    def call(*a, mode=0):
        return lib.sres_resize(*a, mode, None)

    for a in ((None, p) + good[2:], (p, None) + good[2:]):
        assert call(*a) == 1 and b"null pointer" in lib.sres_last_error()
    for i, bad in ((2, 0), (3, 0), (4, -1), (5, 0), (6, -3), (2, -2)):
        a = list(good)
        a[i] = bad
        assert call(*a) == 1 and b"bad shape" in lib.sres_last_error(), (i, bad)
    for mode in (-1, 5, 99):
        assert call(*good, mode=mode) == 1 and b"unknown mode" in lib.sres_last_error()
    for mode in (0, 1, 2, 3):
        for sh, sw in ((0.0, 2.0), (2.0, -1.0), (float("inf"), 2.0), (2.0, float("nan"))):
            assert call(p, p, 2, 8, 8, 4, 4, sh, sw, mode=mode) == 1 and b"scales" in lib.sres_last_error()


def test_torch_interp_mode_maps_the_config_names():
    from sres.base.util.array import torch_interp_mode
    from sres.base.util.config import ConfigContext
    ConfigContext.deactivate()
    ConfigContext.set_defaults(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local")
    expect = {"linear": "bilinear", "cubic": "bicubic", "nearest": "nearest", "nearest-exact": "nearest-exact",
              "area": "area", "bilinear": "bilinear", "bicubic": "bicubic"}
    try:
        for name, torch_name in expect.items():
            with ConfigContext("sres", model="rcan-10-20-64", **{"task.downsample_mode": name, "task.upsample_mode": "cubic"}):
                assert torch_interp_mode(True) == torch_name and torch_interp_mode(False) == "bicubic"
            with ConfigContext("sres", model="rcan-10-20-64", **{"task.downsample_mode": "cubic", "task.upsample_mode": name}):
                assert torch_interp_mode(False) == torch_name and torch_interp_mode(True) == "bicubic"
    finally:
        ConfigContext.deactivate()


@pytest.mark.parametrize("name", ["lanczos", "trilinear", "linear2"])
def test_unknown_mode_raises_value_error(name):
    from sres.base.util.array import _resize
    from sres.base.util.config import ConfigContext
    from sres_b200 import nn as snn
    ConfigContext.deactivate()
    ConfigContext.set_defaults(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local")
    t = torch.zeros(1, 1, 8, 8)          # a CPU tensor: the refusal comes before any device work
    try:
        with ConfigContext("sres", model="rcan-10-20-64", **{"task.downsample_mode": name, "task.upsample_mode": name}):
            for down in (True, False):
                with pytest.raises(ValueError, match="nearest-exact"):
                    _resize(t, 0.25 if down else 4.0, down)
    finally:
        ConfigContext.deactivate()
    with pytest.raises(ValueError, match="nearest-exact"):
        snn.resize(t, 0.25, name)


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _geometries(direction, f):
    """(planes, Hi, Wi): square 48 / 96 / 192 planes, a non-square 37 x 53 plane, 50 x 50 (divisible by 2 only), and the
    training downsample / evaluation upsample at 64 tiles x 16 channels."""
    if direction == "down":
        g = [(3, 192, 192), (5, 96, 96), (7, 48, 48), (2, 37, 53), (4, 50, 50), (1, 50, 50)]
        return g + [(64 * 16, 192, 192)] if f == 4 else g
    g = [(3, 48, 48), (2, 96, 96), (1, 192, 192), (2, 37, 53), (4, 50, 50), (1, 12, 12)]
    return g + [(64 * 16, 48, 48)] if f == 4 else g


def assert_matches_interpolate(got, x, sf, mode, x_dev=None):
    """got (any device) against F.interpolate(x, scale_factor=sf, mode=mode) on the CPU (and, for the nearest modes,
    on the GPU when x_dev is given)."""
    got = got.detach().cpu()
    ref = F.interpolate(x, scale_factor=sf, mode=mode)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if mode in ("nearest", "nearest-exact"):
        assert torch.equal(got, ref)
        if x_dev is not None:
            assert torch.equal(got, F.interpolate(x_dev, scale_factor=sf, mode=mode).cpu())
        return
    mag = F.interpolate(x.abs(), scale_factor=sf, mode=mode)
    err = (got - ref).abs()
    ok = err <= REL * mag
    assert bool(ok.all()), f"{int((~ok).sum())} elements off, worst {float((err / mag.clamp_min(1e-30)).max()):.3e}"


def _run_abi(lib, x_dev, Ho, Wo, sf, mode, misalign=False):
    """sres_resize into a NaN-filled output followed by a guard region; returns the output (the guard is checked)."""
    from sres_b200 import _lib as L
    B, Cc, Hi, Wi = x_dev.shape
    n = B * Cc * Ho * Wo
    if misalign:                         # input 4 bytes past a 16-byte boundary: the row-vector path must not be taken
        store = torch.empty(x_dev.numel() + 1, device=x_dev.device)
        store[1:] = x_dev.reshape(-1)
        xin = store[1:]
        assert xin.data_ptr() % 16 == 4
    else:
        xin = x_dev
    buf = torch.full((n + GUARD,), float("nan"), device=x_dev.device)
    buf[n:] = SENTINEL
    L.check(lib.sres_resize(L.ptr(xin), L.ptr(buf), B * Cc, Hi, Wi, Ho, Wo, 1.0 / sf, 1.0 / sf, L.RESIZE_MODES[mode],
                            L.cur_stream()), "sres_resize")
    torch.cuda.synchronize()
    assert bool((buf[n:] == SENTINEL).all()), "wrote past the output"
    return buf[:n].view(B, Cc, Ho, Wo)


@pytest.mark.gpu
@pytest.mark.parametrize("f", FACTORS)
@pytest.mark.parametrize("direction", ["down", "up"])
@pytest.mark.parametrize("mode", NEW_MODES)
def test_resize_matches_interpolate(lib, mode, direction, f):
    from sres_b200 import nn as snn
    assert torch.cuda.is_available()
    dev = torch.device("cuda:0")
    sf = 1.0 / f if direction == "down" else float(f)
    g = torch.Generator().manual_seed(1000 * f + len(mode) + (7 if direction == "up" else 0))
    for planes, Hi, Wi in _geometries(direction, f):
        Cc = 16 if planes % 16 == 0 else 1
        x = torch.randn(planes // Cc, Cc, Hi, Wi, generator=g)
        x_dev = x.to(dev)
        Ho, Wo = int(math.floor(Hi * sf)), int(math.floor(Wi * sf))
        got = _run_abi(lib, x_dev, Ho, Wo, sf, mode)
        assert_matches_interpolate(got, x, sf, mode, x_dev)
        assert torch.equal(snn.resize(x_dev, sf, mode), got)
        if (planes, Hi) == (3, 192) or (planes, Hi) == (3, 48):
            assert torch.equal(_run_abi(lib, x_dev, Ho, Wo, sf, mode, misalign=True), got)


@pytest.mark.gpu
def test_bicubic_mode_runs_the_bicubic_kernel(lib):
    from sres_b200 import nn as snn
    dev = torch.device("cuda:0")
    x = torch.randn(3, 2, 192, 192, generator=torch.Generator().manual_seed(5)).to(dev)
    for sf in (0.25, 1.0 / 3):
        down = snn.resize(x, sf, "bicubic")
        assert torch.equal(down, snn.bicubic_resize(x, sf))
        assert torch.equal(snn.resize(down, 1.0 / sf, "bicubic"), snn.bicubic_resize(down, 1.0 / sf))


# ---------------------------------------------------------------------------------------------------------------------
# controller level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
TORCH_MODE = {"linear": "bilinear", "nearest": "nearest", "area": "area"}
CONTROLLER_CASES = {
    # name: (downsample_mode, upsample_mode, data_downsample, LR tile size)
    "linear_down_nearest_up": ("linear", "nearest", 1, 12),
    "area_down_linear_up_data_downsample_2": ("area", "linear", 2, 24),
    "nearest_down_linear_up": ("nearest", "linear", 1, 12),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONTROLLER_CASES))
def test_controller_with_interpolation_modes(name, tmp_path):
    """The reference's workflow on the synthetic dataset with non-bicubic modes: apply_network's target and network input
    against F.interpolate, a few training steps on one batch, and the stitched "interpolated" image of process_image (and
    the interpolated tiles of evaluate) against F.interpolate of the input tiles."""
    from sres.base.util.array import upsample
    from sres.base.util.config import ConfigContext
    from sres.controller.config import ResultStructure, TSet
    from sres.controller.workflow import WorkflowController
    from sres.data.tiles import TileIterator
    assert torch.cuda.is_available()
    down, up, dd, tile = CONTROLLER_CASES[name]
    dmode, umode, s = TORCH_MODE[down], TORCH_MODE[up], 4
    ConfigContext.deactivate()
    random.seed(3)
    wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local"), seed=1)
    wc.initialize("sres", "rcan-10-20-64", **{
        "model.nlayers": 2, "model.nblocks": 2, "task.batch_size": 8, "task.lr": 2e-4, "task.tile_size": dict(x=tile, y=tile),
        "task.tile_order": "corrected", "dataset.region": dict(ys=480, xs=480), "dataset.ntimes": 2,
        "task.ttsplit": dict(train=0.5, valid=0.5, test=0.0), "platform.results": str(tmp_path),
        "task.downsample_mode": down, "task.upsample_mode": up, "task.data_downsample": dd})
    try:
        tr = wc.trainer
        assert tr.world == 1
        ctime = tr.get_dataset().get_dset_time_indices()[0]
        batch = tr.get_srbatch(dict(start=0, end=8), ctime)
        hr = batch.data.detach().cpu()
        # apply_network: optional data_downsample pre-step (the target), then the downsample to the network input
        binput, bprod, btarget = tr.apply_network(batch)
        T = tile * s
        assert hr.shape == (8, 2, T, T)
        assert btarget.shape == (8, 2, T // dd, T // dd) and binput.shape == (8, 2, T // dd // s, T // dd // s)
        assert bprod.shape == btarget.shape
        if dd > 1:
            assert_matches_interpolate(btarget, hr, 1.0 / dd, dmode)
        else:
            assert torch.equal(btarget.detach().cpu(), hr)
        assert_matches_interpolate(binput, btarget.detach().cpu(), 1.0 / s, dmode)
        # training steps on that batch: finite and going down
        tr.model.train()
        losses = [tr.train_step(batch).item() for _ in range(6)]
        assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
        # process_image: four products; the interpolated image is the de-normalised upsample of the input tiles
        images, img_losses = wc.inference(0, ResultStructure.Image)
        assert set(images) == {"SSS", "SST"}
        timeslice = tr.load_timeslice(tr.data_timestamps[TSet.Train][0])
        refs, stats = [], []
        with torch.no_grad():
            for ctile in TileIterator.get_iterator(ntiles=timeslice.sizes["tiles"]):
                bd = tr.get_srbatch(ctile, tr.data_timestamps[TSet.Train][0], shuffle=False)
                if bd is None:
                    break
                bi, _, _ = tr.apply_network(bd)
                ref = F.interpolate(bi.detach().cpu(), scale_factor=float(s), mode=umode)
                assert_matches_interpolate(upsample(bi), bi.detach().cpu(), float(s), umode)
                refs.append(dict(interpolated=ref.to(bi.device)))
                stats.append(bd.attrs)
        for ivar, v in enumerate(tr.target_variables):
            im = images[v]
            assert set(im) == {"input", "target", "interpolated", "model"}
            side = 480 // T * T // dd
            assert im["target"].shape == im["model"].shape == im["interpolated"].shape == (side, side)
            assert im["input"].shape == (side // s, side // s)
            assert np.isfinite(img_losses[v]["model"]) and img_losses[v]["interpolated"] > 0
            want = tr.assemble_images(refs, ivar, timeslice.coords["tiles"], timeslice.attrs["grid_shape"], stats)["interpolated"]
            if umode == "nearest":
                np.testing.assert_array_equal(im["interpolated"], want)
            else:
                assert np.nanmax(np.abs(im["interpolated"] - want)) <= 2e-6 * np.nanmax(np.abs(want))
        # evaluate: the interpolated tiles are the upsample of the input tiles it returns
        res, ev_losses = tr.evaluate(TSet.Validation, time_index=0, update_checkpoint=False)
        assert np.isfinite(ev_losses["model"]) and np.isfinite(ev_losses["interpolated"])
        assert_matches_interpolate(torch.from_numpy(res["interpolated"]), torch.from_numpy(res["input"]), float(s), umode)
    finally:
        ConfigContext.deactivate()

