"""Rectangular tiles (task.tile_size {x, y} with x != y) on the GPU: tile extraction, normalisation, the eight flips and
stitching against the CPU oracle; the square entry points unchanged; RCAN / EDSR forward and backward at H != W in both
orientations against the oracle; and the trainer end to end with xyflip alternating the two orientations."""
import os
import random

import numpy as np
import pytest
import torch

import rcan_oracle as O
import tiles_oracle as T
from gpu_util import rel_l2
from synth import sha, synth_hr, synth_region

pytestmark = pytest.mark.gpu
TOL = 1e-2


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda:0")


def _dataset(C_, tile, scale, order, batch_size=7, region=None):
    from sres.base.util.config import ConfigContext
    from sres.data.batch import BatchDataset
    ConfigContext.deactivate()
    ConfigContext.set_defaults(task="SSS_SST-tiles-48" if C_ == 2 else "SST-tiles-48", dataset="synthetic_1200", platform="local")
    dfs = {2: [2], 4: [2, 2]}[scale]
    cc = ConfigContext.activate_global("sres", model="rcan-10-20-64", **{
        "task.batch_size": batch_size, "task.tile_size": dict(tile), "task.tile_order": order,
        "model.downscale_factors": dfs, "model.nlayers": 1, "model.nblocks": 1})
    return cc, BatchDataset(region_source=(lambda t: region) if region is not None else None)


def _region(C_, Y, X, seed, same_mask):
    var = synth_region(C_, Y, X, seed)
    if C_ > 1 and same_mask:
        # the other variables take variable 0's land mask; their own land is filled with noise, not a constant: a
        # constant tile has std 0 and normalises to 0/0, whose NaN bit pattern differs between the host and the GPU
        rng = np.random.default_rng(seed)
        m = np.isnan(var[0])
        for v in var[1:]:
            hole = np.isnan(v)
            v[hole] = 0.5 + rng.standard_normal(int(hole.sum())).astype(np.float32)
            v[m] = np.nan
    return var


# (C, tile_size, scale, order); the regions are sized so that neither axis is a multiple of the HR tile
TILE_CASES = [
    (1, dict(x=12, y=7), 4, "reference"),
    (1, dict(x=7, y=12), 2, "reference"),
    (2, dict(x=12, y=7), 2, "reference"),
    (2, dict(x=7, y=12), 4, "reference"),
    (2, dict(x=12, y=7), 4, "corrected"),
    (2, dict(x=7, y=12), 2, "corrected"),
]


@pytest.mark.parametrize("C_,tile,scale,order", TILE_CASES)
def test_rect_tiles_extract_norm_flip_stitch(C_, tile, scale, order, dev):
    from sres.base.util.config import ConfigContext
    from sres.controller.dual_trainer import ModelTrainer
    Y, X = 333, 517
    var = _region(C_, Y, X, seed=31 + C_ + scale, same_mask=(order == "reference"))
    region = np.concatenate(var, 0)
    cc, ds = _dataset(C_, tile, scale, order, region=region)
    try:
        ts = ds.load_timeslice(0)
        tiles_o, ids_o, gs_o = T.get_tiles(var, tile, scale, mode=order)
        Th, Tw = tile["y"] * scale, tile["x"] * scale
        assert Y % Th and X % Tw
        assert ts.shape == tiles_o.shape and ts.shape[2:] == (Th, Tw) and ts.shape[0] >= 14
        assert sha(ts.values) == sha(tiles_o)
        np.testing.assert_array_equal(ts.coords["tiles"], ids_o)
        assert ts.attrs["grid_shape"] == gs_o
        # lnorm within the square tests' bounds; flips: exact permutations of the unflipped normalised batch
        nb = ds.select_batch((7, 14))
        nb_o, st_o = T.lnorm(T.select_batch(tiles_o, 7, 14))
        np.testing.assert_allclose(nb.values, nb_o, rtol=0, atol=2e-5)
        np.testing.assert_allclose(nb.attrs["mean"].cpu().numpy(), st_o["mean"], rtol=1e-6)
        np.testing.assert_allclose(nb.attrs["std"].cpu().numpy(), st_o["std"], rtol=1e-5)
        base = nb.values
        for fi in range(8):
            fb = ds.norm(ts.data[7:14], (7, 14), fi)
            assert fb.shape == ((7, C_, Tw, Th) if fi >= 4 else (7, C_, Th, Tw))
            np.testing.assert_array_equal(fb.values, T.xyflip(base, fi))
        # stitching: raw tiles, and normalised tiles de-normalised by the kernel, against assemble_images (+ denorm)
        tr = object.__new__(ModelTrainer)
        tr.device = dev
        raw_o, raw_g, nrm_o, nrm_g, stats = [], [], [], [], []
        for b in T.tile_batches(tiles_o.shape[0], 7):
            raw = T.select_batch(tiles_o, b["start"], b["end"])
            raw_o.append(dict(target=raw, input=np.ascontiguousarray(raw[:, :, ::scale, ::scale])))
            raw_g.append({k: torch.from_numpy(v).to(dev) for k, v in raw_o[-1].items()})
            bd, st = T.lnorm(raw)
            bd_in = np.ascontiguousarray(bd[:, :, ::scale, ::scale])
            nrm_o.append(dict(target=T.denorm(bd, st), input=T.denorm(bd_in, st)))
            nrm_g.append(dict(target=torch.from_numpy(bd).to(dev), input=torch.from_numpy(bd_in).to(dev)))
            stats.append({k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in st.items()})
        for ivar in range(C_):
            for got, want in ((tr.assemble_images(raw_g, ivar, ts.coords["tiles"], ts.attrs["grid_shape"]),
                               T.assemble_images(raw_o, ivar, ids_o, gs_o)),
                              (tr.assemble_images(nrm_g, ivar, ts.coords["tiles"], ts.attrs["grid_shape"], stats),
                               T.assemble_images(nrm_o, ivar, ids_o, gs_o))):
                assert got["target"].shape == (gs_o["y"] * Th, gs_o["x"] * Tw)
                assert got["input"].shape == (gs_o["y"] * Th // scale, gs_o["x"] * Tw // scale)
                for k in want:
                    assert got[k].dtype == want[k].dtype and sha(got[k]) == sha(want[k]), (ivar, k)
    finally:
        ConfigContext.deactivate()


def test_square_entry_points_equal_rectangular_ones(dev):
    """The square entry points are the rectangular ones with Th = Tw = T: byte-identical outputs for all four kernels and
    all eight flips."""
    from sres_b200 import _lib as L
    lib = L.lib()
    g = torch.Generator().manual_seed(7)
    Cc, Y, X, Tt, gy, gx = 2, 150, 170, 24, 5, 6
    region = torch.randn(Cc, Y, X, generator=g)
    region[:, 20:40, 30:75] = float("nan")
    region = region.to(dev)
    ncand = Cc * gy * gx
    st = L.cur_stream()
    f_sq = torch.empty(ncand, dtype=torch.int32, device=dev)
    f_hw = torch.empty_like(f_sq)
    L.check(lib.sres_tiles_finite_flags(L.ptr(region), Cc, Y, X, 3, 5, Tt, gy, gx, L.ptr(f_sq), st), "flags")
    L.check(lib.sres_tiles_finite_flags_hw(L.ptr(region), Cc, Y, X, 3, 5, Tt, Tt, gy, gx, L.ptr(f_hw), st), "flags_hw")
    assert torch.equal(f_sq, f_hw) and 0 < int(f_sq.sum()) < ncand
    src = torch.arange(ncand, dtype=torch.int32, device=dev).flip(0).contiguous()
    t_sq = torch.empty(ncand, Tt, Tt, device=dev)
    t_hw = torch.empty_like(t_sq)
    L.check(lib.sres_tiles_gather(L.ptr(region), Cc, Y, X, 3, 5, Tt, gy, gx, L.ptr(src), ncand, L.ptr(t_sq), st), "gather")
    L.check(lib.sres_tiles_gather_hw(L.ptr(region), Cc, Y, X, 3, 5, Tt, Tt, gy, gx, L.ptr(src), ncand, L.ptr(t_hw), st),
            "gather_hw")
    assert sha(t_sq.cpu().numpy()) == sha(t_hw.cpu().numpy())
    for fi in range(8):
        outs = []
        for hw in (False, True):
            o, m, s = torch.empty_like(t_sq), torch.empty(ncand, device=dev), torch.empty(ncand, device=dev)
            if hw:
                L.check(lib.sres_tiles_lnorm_hw(L.ptr(t_sq), ncand, Tt, Tt, fi, L.ptr(o), L.ptr(m), L.ptr(s), st), "lnorm_hw")
            else:
                L.check(lib.sres_tiles_lnorm(L.ptr(t_sq), ncand, Tt, fi, L.ptr(o), L.ptr(m), L.ptr(s), st), "lnorm")
            outs.append([sha(x.cpu().numpy()) for x in (o, m, s)])
        assert outs[0] == outs[1], fi
    tiles = t_sq.reshape(ncand // Cc, Cc, Tt, Tt)
    cell = torch.full((gy * gx,), -1, dtype=torch.int32, device=dev)
    cell[: ncand // Cc - 3] = torch.arange(ncand // Cc - 3, dtype=torch.int32, device=dev)
    mean = torch.rand(ncand, device=dev)
    std = torch.rand(ncand, device=dev) + 0.5
    for mp, sp in ((None, None), (mean, std)):
        i_sq = torch.empty(gy * Tt, gx * Tt, device=dev)
        i_hw = torch.empty_like(i_sq)
        L.check(lib.sres_tiles_stitch(L.ptr(tiles), Cc, 1, Tt, gy, gx, L.ptr(cell), L.ptr(mp), L.ptr(sp), L.ptr(i_sq), st), "stitch")
        L.check(lib.sres_tiles_stitch_hw(L.ptr(tiles), Cc, 1, Tt, Tt, gy, gx, L.ptr(cell), L.ptr(mp), L.ptr(sp), L.ptr(i_hw), st),
                "stitch_hw")
        assert sha(i_sq.cpu().numpy()) == sha(i_hw.cpu().numpy())


# ------------------------------------------------------------------------------------------------
# the model at H != W
# ------------------------------------------------------------------------------------------------
def _rect_hr(B, C_, Hh, Wh, seed=4456):
    """Smooth, per-tile normalised HR batch (like lnorm'd ocean tiles) of shape (B, C, Hh, Wh)."""
    x = synth_hr(B, C_, max(Hh, Wh), seed=seed, smooth=True)[:, :, :Hh, :Wh]
    return ((x - x.mean((2, 3), keepdim=True)) / x.std((2, 3), keepdim=True)).contiguous()


def _build(cfg, C_, dev_):
    from sres_b200 import nn as snn
    if O.is_edsr(cfg):
        return snn.EDSR(nchannels_in=C_, nchannels_out=C_, nfeatures=64, nlayers=cfg["nlayers"], scale=O.scale_of(cfg),
                        res_scale=cfg["res_scale"], device=dev_)
    return snn.RCAN(nchannels_in=C_, nchannels_out=C_, nfeatures=64, nlayers=cfg["nlayers"], nblocks=cfg["nblocks"],
                    cbottleneck=cfg["cbottleneck"], scale=O.scale_of(cfg), device=dev_)


# name: (cfg overrides, B, channels, LR (H, W))
MODEL_CASES = {
    "rcan_x4_7x12": (dict(nlayers=2, nblocks=2), 2, 2, (7, 12)),
    "rcan_x4_12x7": (dict(nlayers=2, nblocks=2), 2, 2, (12, 7)),
    "rcan_x3_10x16": (dict(nlayers=1, nblocks=2, downscale_factors=[3]), 2, 2, (10, 16)),
    "edsr_x2_20x9": (dict(name="edsr", nlayers=2, downscale_factors=[2]), 2, 2, (20, 9)),
    "rcan_x8_4ch_6x24": (dict(nlayers=1, nblocks=1, downscale_factors=[2, 2, 2]), 1, 4, (6, 24)),
    "rcan_x2_4x130": (dict(nlayers=1, nblocks=2, downscale_factors=[2]), 2, 1, (4, 130)),
    "rcan_x2_130x4": (dict(nlayers=1, nblocks=2, downscale_factors=[2]), 2, 1, (130, 4)),
}


@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_rect_model_matches_oracle(name, dev):
    from sres_b200 import nn as snn
    over, B, C_, (H, W) = MODEL_CASES[name]
    cfg = O.model_cfg(**over)
    scale = O.scale_of(cfg)
    sd = O.make_state_dict(cfg, C_, C_)
    hr = _rect_hr(B, C_, H * scale, W * scale)
    loss_o, prd_o, grads_o = O.loss_and_grads(hr, sd, cfg, "l2")
    model = _build(cfg, C_, dev)
    model.load_state_dict(sd)
    hr_d = hr.to(dev)
    lr_d = snn.bicubic_resize(hr_d, 1.0 / scale)
    assert lr_d.shape == (B, C_, H, W)
    prd = model(lr_d.requires_grad_(True))
    loss = snn.loss(prd, hr_d, "l2")
    loss.backward()
    assert prd.shape == (B, C_, H * scale, W * scale)
    ro = rel_l2(prd.detach().cpu(), prd_o)
    num = sum((p.grad.cpu() - grads_o[k]).double().pow(2).sum().item() for k, p in model.named_parameters())
    den = sum(g.double().pow(2).sum().item() for g in grads_o.values())
    rg = (num / den) ** 0.5
    print(f"{name}: output rel-L2 {ro:.3e}, gradient rel-L2 {rg:.3e}, loss {loss.item():.6f} vs {loss_o:.6f}")
    assert ro < TOL and rg < TOL and abs(loss.item() - loss_o) < TOL * abs(loss_o)
    with torch.no_grad():
        assert rel_l2(model(lr_d.detach()).cpu(), prd_o) < TOL        # inference mode (its own workspace)


def test_orientation_selects_the_launch_path(dev):
    """At LR 4 x 130 the rows are too long for the fused convolution pair (W + 2 > 128) and the x2 tail runs on the
    wide-image CUDA-core kernel; at 130 x 4 both take the tensor-core paths.  The library's kernel count per forward tells
    them apart (the fused pair is one launch for two convolutions)."""
    cfg = O.model_cfg(nlayers=1, nblocks=2, downscale_factors=[2])
    model = _build(cfg, 1, dev)
    model.load_state_dict(O.make_state_dict(cfg, 1, 1))
    with torch.no_grad():
        for H, W in ((4, 130), (130, 4)):
            model(torch.randn(2, 1, H, W, device=dev))
    wide, tall = model.engine.launches_forward(4, 130, False), model.engine.launches_forward(130, 4, False)
    print(f"kernels per forward: LR 4 x 130 {wide}, LR 130 x 4 {tall}")
    assert tall < wide


def test_orientations_alternate_in_one_engine_with_graphs(dev):
    """(B, h, w), then (B, w, h), then (B, h, w) again in one engine with CUDA graphs on (the first call of a shape runs
    eagerly, later ones replay captured graphs): with no optimizer step in between, the third pass reproduces the first
    bit for bit, output and every gradient."""
    from sres_b200 import nn as snn
    assert os.environ.get("SRES_CUDA_GRAPHS", "1") != "0"
    cfg = O.model_cfg(nlayers=2, nblocks=2)
    sd = O.make_state_dict(cfg, 2, 2)
    model = _build(cfg, 2, dev)
    model.load_state_dict(sd)
    h, w = 7, 12

    def run(H, W):
        hr = _rect_hr(4, 2, H * 4, W * 4, seed=9).to(dev)
        model.zero_grad(set_to_none=True)
        prd = model(snn.bicubic_resize(hr, 0.25).requires_grad_(True))
        snn.loss(prd, hr, "l2").backward()
        torch.cuda.synchronize()
        return prd.detach().clone(), model.engine.flat_grad.detach().clone()

    first = run(h, w)
    other = run(w, h)
    third = run(h, w)
    assert other[0].shape == (4, 2, w * 4, h * 4)
    assert torch.equal(first[0], third[0]) and torch.equal(first[1], third[1])
    assert model.engine._graphs.get(("fwd", (4, h, w, True))) is not None
    assert model.engine._graphs[("bwd", (4, h, w, True), False, 0, model.engine.num_segments())]["graph"] is not None


def test_shape_cache_keeps_both_orientations_together(dev):
    """A shape and its transpose are one entry of the engine's workspace cache: with MAX_SHAPES entries in use, touching
    either orientation keeps both, and a new entry evicts both orientations of the least recently used one."""
    from sres_b200.engine import RcanEngine
    eng = RcanEngine(2, 2, 64, 1, 1, 2, 2, dev)
    allocs = []
    evict = eng._evict_shapes
    eng._evict_shapes = lambda key: (allocs.append(key), evict(key))
    n = eng.MAX_SHAPES
    keys = []
    for b in range(1, n + 1):                       # n entries, two orientations each
        keys += [(b, 6, 10, True), (b, 10, 6, True)]
    for k in keys:
        eng.workspace(*k)
    assert len(allocs) == 2 * n and set(eng._ws) == set(keys)
    for k in keys:                                  # steady state: every orientation of every entry stays resident
        eng.workspace(*k)
    assert len(allocs) == 2 * n
    eng.workspace(1, 10, 6, True)                   # entry 1 becomes the most recent (through its other orientation)
    eng.workspace(n + 1, 6, 10, True)               # a new entry evicts entry 2, both orientations
    assert (2, 6, 10, True) not in eng._ws and (2, 10, 6, True) not in eng._ws
    assert (1, 6, 10, True) in eng._ws and (1, 10, 6, True) in eng._ws and len(eng._ws) == 2 * n - 1


def test_workspace_per_orientation_is_separate(dev):
    """The two orientations never share a workspace (the padding rows of the PixelUnshuffle-layout gradient buffers are
    different rows)."""
    from sres_b200.engine import RcanEngine
    eng = RcanEngine(2, 2, 64, 1, 1, 2, 4, dev)
    a, b = eng.workspace(4, 7, 12, True), eng.workspace(4, 12, 7, True)
    assert a.data_ptr() != b.data_ptr()


# ------------------------------------------------------------------------------------------------
# the trainer with xyflip alternating the orientations
# ------------------------------------------------------------------------------------------------
def _clean_region(t):
    """(2, 112, 768) NaN-free region: 4 x 16 tiles of 28 x 48, every one survives, so each timeslice holds 64 tiles."""
    yy, xx = np.meshgrid(np.arange(112, dtype=np.float32), np.arange(768, dtype=np.float32), indexing="ij")
    rng = np.random.default_rng(100 + t)
    out = np.stack([np.sin(xx / 23.0 + c + t) * np.cos(yy / 17.0) * (3.0 + c) + 20.0 * (c + 1) for c in range(2)])
    return (out + rng.standard_normal(out.shape).astype(np.float32) * 0.1).astype(np.float32)


def test_trainer_with_rect_tiles_and_xyflip(dev, tmp_path, monkeypatch):
    from sres.base.util.config import ConfigContext, cfg
    from sres.controller.config import TSet
    from sres.controller.workflow import WorkflowController
    from sres.data.batch import BatchDataset
    ConfigContext.deactivate()
    random.seed(5)
    wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local"), seed=1)
    wc.initialize("sres", "rcan-10-20-64", **{
        "model.nlayers": 1, "model.nblocks": 1, "task.batch_size": 4, "task.lr": 2e-4, "task.tile_size": dict(x=12, y=7),
        "task.xyflip": True, "task.tile_order": "corrected", "dataset.ntimes": 4,
        "task.ttsplit": dict(train=0.5, valid=0.5, test=0.0), "platform.results": str(tmp_path)})
    try:
        tr = wc.trainer
        tr.model_manager._dataset = BatchDataset(region_source=_clean_region)
        eng = tr.model.engine
        counts = dict(alloc=0, capture=0)
        evict = eng._evict_shapes

        def counting_evict(key):
            counts["alloc"] += 1
            return evict(key)
        eng._evict_shapes = counting_evict

        class CountingGraph(torch.cuda.CUDAGraph):
            def capture_begin(self, *a, **k):
                counts["capture"] += 1
                return super().capture_begin(*a, **k)
        monkeypatch.setattr(torch.cuda, "CUDAGraph", CountingGraph)
        at_save, shapes = [], []
        save = tr.checkpoint_manager.save_checkpoint

        def counting_save(*a, **k):
            at_save.append(dict(counts))
            return save(*a, **k)
        tr.checkpoint_manager.save_checkpoint = counting_save
        apply = tr.apply_network

        def recording_apply(batch):
            if tr.model.training:
                shapes.append((len(at_save), tuple(batch.shape)))
            return apply(batch)
        tr.apply_network = recording_apply

        out = tr.train(2, True, seed=4456, interp_loss=True, verbose=False)     # epochs [1, 2): one epoch
        assert np.isfinite(out["prediction"])
        # both orientations ran at least twice in the first timeslice (first call eager, second captured) ...
        first = [s for i, s in shapes if i == 0]
        assert len(first) == 16 and first.count((4, 2, 28, 48)) >= 2 and first.count((4, 2, 48, 28)) >= 2, first
        assert {s for i, s in shapes if i == 1} <= {(4, 2, 28, 48), (4, 2, 48, 28)}
        # ... so the second timeslice allocated no workspace and captured no graph (saves 1 and 2 close the two training
        # timeslices; the epoch-end validation pass may write a third)
        assert len(at_save) >= 2 and at_save[0]["alloc"] == 2 and at_save[1] == at_save[0], at_save
        assert [h["epoch"] for h in tr.eval_history[TSet.Validation]] == [1]

        # inference: per-axis image sizes, and the model image is the per-tile products placed by the oracle
        images, losses = tr.process_image(TSet.Train, 0)
        gs = tr.get_dataset().timeslice.attrs["grid_shape"]
        assert gs == dict(y=4, x=16)
        for v in images:
            assert images[v]["target"].shape == (4 * 28, 16 * 48) and images[v]["input"].shape == (4 * 7, 16 * 12)
            assert np.isfinite(losses[v]["model"])
        ts = tr.get_dataset().timeslice
        prods, stats = [], []
        with torch.no_grad():
            for ctile in T.tile_batches(ts.shape[0], 4):
                bd = tr.get_srbatch(ctile, tr.get_dataset().time_index)
                assert bd.attrs["xyflip"] == 0
                _, prd, _ = tr.apply_network(bd)
                prods.append(dict(model=T.denorm(prd.cpu().numpy(), {k: bd.attrs[k].cpu().numpy() for k in ("mean", "std")})))
        for ivar, v in enumerate(tr.target_variables):
            want = T.assemble_images(prods, ivar, ts.coords["tiles"], gs)["model"]
            assert images[v]["model"].dtype == want.dtype and sha(images[v]["model"]) == sha(want), v

        # evaluate(keep_results=True): two tile shapes cannot be concatenated with xyflip on; arrays with it off
        cfg().task["xyflip"] = True
        with pytest.raises(ValueError, match="xyflip"):
            tr.evaluate(TSet.Validation, time_index=0)
        cfg().task["xyflip"] = False
        res, l2 = tr.evaluate(TSet.Validation, time_index=0)
        assert res["model"].shape[1:] == (2, 28, 48) and res["input"].shape[1:] == (2, 7, 12) and np.isfinite(l2["model"])
    finally:
        ConfigContext.deactivate()
