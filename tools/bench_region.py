"""Config 4 (SURVEY 8d): inference over a whole region through the mirrored controller API -- extract tiles, lnorm,
bicubic down, RCAN-full forward (no grad), denorm, stitch -- on the synthetic stand-in for the swot_20-20e roi
(3000 x 17280, 15 x 90 grid, 1350 tiles per variable, ~20 % land).  Also times one EDSR-16 and one RCAN-full training
step for the record.  Prints output megapixels per second (36 864 px per tile and variable).

    python tools/bench_region.py                                   # 48 x 48 tiles, as above
    python tools/bench_region.py --tiles 48x48,48x50,64x36,36x64 --train-tiles 48x48,64x36,36x64

--tiles: task.tile_size values written XxY (LR pixels, x then y; the HR tile is 4x that).  For each: region inference
passes, and the tile-path kernels (NaN-tile flags, gather, lnorm, stitch) over the whole region in GB/s.
--train-tiles: RCAN-full x4 training steps at LR batches (64, 2, y, x), the shapes taking turns on one model; median
step time and the model's kernels per step in each shape."""
import argparse, ctypes as C, os, subprocess, sys, tempfile, time
import numpy as np, torch
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "super-resolution-climate_b200"))
from sres.base.util.config import ConfigContext
from sres.controller.config import ResultStructure
from sres.controller.workflow import WorkflowController
from sres_b200 import _lib as L
from sres_b200 import nn as snn

dev = torch.device("cuda:0")
tmp = tempfile.mkdtemp()


def _tile_list(arg):
    return [dict(x=int(a), y=int(b)) for a, b in (t.split("x") for t in arg.split(","))] if arg else []


ap = argparse.ArgumentParser()
ap.add_argument("--tiles", default="")
ap.add_argument("--train-tiles", default="")
args = ap.parse_args()
if args.tiles or args.train_tiles:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
    print(f"card: {card}")


def region_inference(tile, reps=3):
    """Median of `reps` region passes through the controller API at one tile size, and the controller for reuse."""
    ConfigContext.deactivate()
    wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_20-20e", platform="local"), seed=1)
    wc.initialize("sres", "rcan-10-20-64", **{"model.cbottleneck": 16, "task.batch_size": 64, "task.tile_order": "corrected",
                                               "task.tile_size": dict(tile), "dataset.ntimes": 2, "platform.results": tmp})
    th, tw = tile["y"] * 4, tile["x"] * 4
    wc.inference(0, ResultStructure.Image)                       # warm-up: workspaces, graphs, the ragged last batch
    dts = []
    for rep in range(reps):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        images, _ = wc.inference(0, ResultStructure.Image)
        torch.cuda.synchronize(); dts.append(time.perf_counter() - t0)
    img = images["SSS"]["model"]
    ntiles = int(np.isfinite(img[::th, ::tw]).sum())
    dt = float(np.median(dts))
    mp = 2 * ntiles * th * tw / 1e6
    rows = img.shape[0]
    print(f"tile_size x={tile['x']} y={tile['y']} (HR {th} x {tw}): region inference median of {reps} passes {dt:.3f} s, "
          f"{ntiles} tiles x 2 vars, image {img.shape} ({rows} of 3000 ROI rows tiled) -> {mp / dt:.1f} output MP/s end to end "
          f"(host images included)")
    return wc


def tile_kernels(wc, tile, reps=20):
    """The tile-path kernels over the whole region (2 x 3000 x 17280 fp32 = 415 MB, larger than L2), CUDA events around
    `reps` launches each.  GB/s counts the bytes each kernel has to move once: the candidate tiles read (flags), tiles
    read + written (gather, lnorm), tiles read + image written (stitch, one variable)."""
    ds = wc.trainer.get_dataset()
    lib = L.lib()
    region = ds._load_region_on_device(0)
    Cc, Y, X = region.shape
    Th, Tw = tile["y"] * 4, tile["x"] * 4
    gs = ds.tile_grid.get_grid_shape(image_shape=dict(c=Cc, y=Y, x=X))
    gy, gx = gs["y"], gs["x"]
    ncand = gy * gx
    flags = torch.empty(Cc * ncand, dtype=torch.int32, device=dev)
    src = torch.arange(Cc * ncand, dtype=torch.int32, device=dev).reshape(Cc, ncand).t().contiguous()
    tiles = torch.empty(ncand, Cc, Th, Tw, device=dev)
    normed = torch.empty_like(tiles)
    mean = torch.empty(ncand * Cc, device=dev)
    std = torch.empty_like(mean)
    cell = torch.arange(ncand, dtype=torch.int32, device=dev)
    img = torch.empty(gy * Th, gx * Tw, device=dev)
    st = L.cur_stream()
    tile_bytes = ncand * Cc * Th * Tw * 4
    calls = {
        "finite_flags": (lambda: lib.sres_tiles_finite_flags_hw(L.ptr(region), Cc, Y, X, 0, 0, Th, Tw, gy, gx, L.ptr(flags), st),
                         tile_bytes),
        "gather": (lambda: lib.sres_tiles_gather_hw(L.ptr(region), Cc, Y, X, 0, 0, Th, Tw, gy, gx, L.ptr(src), ncand * Cc,
                                                    L.ptr(tiles), st), 2 * tile_bytes),
        "lnorm (flip 5)": (lambda: lib.sres_tiles_lnorm_hw(L.ptr(tiles), ncand * Cc, Th, Tw, 5, L.ptr(normed), L.ptr(mean),
                                                           L.ptr(std), st), 2 * tile_bytes),
        "stitch + denorm": (lambda: lib.sres_tiles_stitch_hw(L.ptr(tiles), Cc, 0, Th, Tw, gy, gx, L.ptr(cell), L.ptr(mean),
                                                             L.ptr(std), L.ptr(img), st), 2 * tile_bytes // Cc),
    }
    out = []
    for name, (fn, nbytes) in calls.items():
        L.check(fn(), name)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / reps * 1e-3
        out.append(f"{name} {t * 1e6:.0f} us {nbytes / t / 1e9:.0f} GB/s ({nbytes / t / 1e9 / 6545:.0%} of 6545)")
    print(f"  tile kernels, {gy} x {gx} tiles x {Cc} vars: " + "; ".join(out))


def train_alternating(train_tiles, nsteps=30, B=64):
    """RCAN-full x4 training steps, the LR shapes (B, 2, y, x) taking turns on one model: median step time per shape over
    `nsteps` rounds (CUDA events), and the model's kernels per step in each shape (forward + backward, counted by the
    library through sres_launch_count)."""
    ConfigContext.deactivate()
    model = snn.RCAN(nchannels_in=2, nchannels_out=2, nfeatures=64, nlayers=10, nblocks=20, cbottleneck=16, scale=4, device=dev)
    opt = snn.FusedAdam(model, lr=1e-4)
    shapes = [(t["y"], t["x"]) for t in train_tiles]
    hrs = {s: torch.randn(B, 2, s[0] * 4, s[1] * 4, device=dev) for s in shapes}
    times = {s: [] for s in shapes}
    kernels = {}
    for it in range(nsteps + 3):
        for s in shapes:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0 = model.engine.launches
            e0.record()
            opt.zero_grad()
            snn.loss(model(snn.bicubic_resize(hrs[s], 0.25).requires_grad_(True)), hrs[s], "l2").backward()
            opt.step()
            e1.record()
            kernels[s] = model.engine.launches - n0
            if it >= 3:                                  # the first calls of a shape run eagerly, then capture graphs
                torch.cuda.synchronize()
                times[s].append(e0.elapsed_time(e1))
    ws = {s: model.engine._ws[(B, s[0], s[1], True)].numel() for s in shapes}
    for s in shapes:
        print(f"RCAN-full x4 train step, B={B}, LR {s[0]} x {s[1]} (H x W): median {np.median(times[s]):.2f} ms "
              f"(min {min(times[s]):.2f}, max {max(times[s]):.2f}, {len(times[s])} steps), {kernels[s]} model kernels per step, "
              f"workspace {ws[s] / 2**30:.2f} GiB")


if args.tiles or args.train_tiles:
    for tile in _tile_list(args.tiles):
        wc = region_inference(tile)
        tile_kernels(wc, tile)
        del wc
        torch.cuda.empty_cache()
    if args.train_tiles:
        train_alternating(_tile_list(args.train_tiles))
    sys.exit(0)

wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_20-20e", platform="local"), seed=1)
wc.initialize("sres", "rcan-10-20-64", **{"model.cbottleneck": 16, "task.batch_size": 64, "task.tile_order": "corrected",
                                           "dataset.ntimes": 2, "platform.results": tmp})
for rep in range(3):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    images, losses = wc.inference(0, ResultStructure.Image)
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    img = images["SSS"]["model"]
    ntiles = int(np.isfinite(img[::192, ::192]).sum())
    mp = 2 * ntiles * 192 * 192 / 1e6
    print(f"region inference pass {rep}: {dt:.3f} s, {ntiles} tiles x 2 vars, image {img.shape} -> {mp / dt:.1f} output MP/s end to end "
          f"(host images included)")
ConfigContext.deactivate()

def step_time(model, B=64, n=8):
    opt = snn.FusedAdam(model, lr=1e-4)
    hr = torch.randn(B, 2, 192, 192, device=dev)
    for it in range(n + 3):
        if it == 3:
            torch.cuda.synchronize(); t0 = time.perf_counter()
        opt.zero_grad()
        snn.loss(model(snn.bicubic_resize(hr, 0.25).requires_grad_(True)), hr, "l2").backward()
        opt.step()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n

edsr = snn.EDSR(nchannels_in=2, nchannels_out=2, nfeatures=64, nlayers=16, scale=4, device=dev)
t = step_time(edsr)
print(f"EDSR-16 x4 train step, B=64: {t * 1e3:.2f} ms = {64 / t:.0f} tiles/s")
with torch.no_grad():
    x = torch.randn(64, 2, 48, 48, device=dev)
    for _ in range(3): edsr(x)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(20): edsr(x)
    torch.cuda.synchronize(); t = (time.perf_counter() - t0) / 20
print(f"EDSR-16 x4 forward, B=64: {t * 1e3:.2f} ms = {64 / t:.0f} tiles/s = {64 / t * 36864 / 1e6:.0f} output MP/s")
