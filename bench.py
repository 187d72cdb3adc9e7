#!/usr/bin/env python
"""Benchmark of the RCAN hot path (BASELINE.json metric: RCAN train tiles/s, 48x48 2-ch, x4).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] ...                # the reference's own CPU path (oracle/_ref, else the port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # data parallel, one rank per GPU

One step = one optimizer step of RCAN-full (10 groups x 20 RCABs, 64 features, reduction 16, x4) on a
batch of 64 synthetic 2-channel 48x48 LR tiles per GPU: bicubic down of the HR batch, forward, RMSE
loss, backward, fused Adam.  Prints ONE JSON line (rank 0).  Besides the headline (BASELINE config 2 / 3) the line
carries `infer_region` (config 4: tile extraction, batched forward, stitching of a 3000 x 17280 region, host images out)
and `x8` (config 5: x8 upscaling of 4-channel 96 x 96 tiles); `--skip-extras` leaves them out.

`--dump-outputs DIR` (CUDA arm, rank 0) writes what the last timed training step computed to DIR/*.npy, float32:
`loss` (what train_step returned), `prediction` (the model output it was computed from, 64 x 2 x 192 x 192), and
`params_sample` / `grads_sample` (the updated parameters and their gradients at a fixed, seeded set of 2^20 of the
16.3 M flat indices).  Inputs and initial weights are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "super-resolution-climate_b200")   # put on sys.path by the CUDA arm only: the reference arm imports the
                                                            # reference's own `sres` package, which has the same name

WORKLOAD = dict(nlayers=10, nblocks=20, nfeatures=64, cbottleneck=16, downscale_factors=[2, 2])
TILE, CH, SCALE, BATCH = 48, 2, 4, 64
METRIC = "rcan_train_tiles_per_s"


def flops_per_tile(train=True):
    """Algorithmic FLOPs per LR tile (BASELINE.md section 4): 2*MACs of all convolutions + CA MLP."""
    Fn, G, R, red, S, s = 64, WORKLOAD["nlayers"], WORKLOAD["nblocks"], WORKLOAD["cbottleneck"], TILE, SCALE
    ups = 4 * Fn * Fn * 1 + 4 * Fn * Fn * 4
    fwd = 2 * 9 * S * S * (CH * Fn + (G * (2 * R + 1) + 1) * Fn * Fn + ups + Fn * CH * s * s) + G * R * 4 * Fn * Fn / red
    return fwd * (3 if train else 1)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops_burst=p["bf16_tflops"], tflops_sustained=p["bf16_tflops_sustained"], hbm=p["hbm_gbs"], src="measured")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx, self.samples, self.reasons, self.max_mhz, self._halt = gpu_index, [], set(), None, threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons))


def synth_hr(B, C, S, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, C, S, S, generator=g)


DUMP_SAMPLE = 1 << 20   # parameters / gradients sampled per dump: the full flat buffers are 65 MB each


def dump_outputs(dirname, loss, prediction, eng):
    """Write the last training step's results as float32 .npy files (see the module docstring)."""
    import numpy as np
    import torch
    idx = torch.randperm(eng.n_params, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    idx = idx.to(eng.flat.device)
    arrays = {"loss": loss.reshape(1), "prediction": prediction, "params_sample": eng.flat[idx], "grads_sample": eng.flat_grad[idx]}
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's OWN code (oracle/_ref = byte-for-byte staged copy of its `sres`
# package, oracle/make_ref.py) on the host cores; the oracle port only when no copy of the reference is around
# ---------------------------------------------------------------------------------------------------
CPU_WORKLOADS = {
    # name: (model overrides, sample batch) -- BASELINE.md 5.3: RCAN-full on CPU is timed at batch 4..8
    "full": (WORKLOAD, 8),
    "config1": (dict(nlayers=4, nblocks=4, nfeatures=64, cbottleneck=16, downscale_factors=[2, 2]), 16),
}


def reference_step_fn(overrides, batch):
    """(kind, step): one optimizer step of the reference's train loop body (dual_trainer.py:310-323 without logging)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import rcan_oracle as O
    import ref_import as R
    cfg = O.model_cfg(**overrides)
    hr = synth_hr(batch, CH, TILE * SCALE, 4456)
    if R.available():
        from synth import TASK
        R.set_cfg(cfg, TASK)
        import importlib
        get_model = importlib.import_module(f"sres.model.{cfg['name']}.network").get_model      # manager.py:93-95
        from sres.base.util import array as ref_array
        from sres.controller.stats import l2loss as ref_l2
        import sres.base.gpu as ref_gpu
        ref_gpu.get_device = lambda: torch.device("cpu")
        ref_array.get_device = ref_gpu.get_device
        torch.manual_seed(4456)
        model = get_model(nchannels_in=CH, nchannels_out=CH, device=torch.device("cpu"))
        model.train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=0.0)                      # dual_trainer.py:126

        def step():
            opt.zero_grad()
            target = hr.clone().requires_grad_(True)        # array2tensor: requires_grad=True (array.py:70)
            prd = model(ref_array.downsample(target))       # dual_trainer.py:569-570
            loss = ref_l2(prd, target)
            loss.backward()
            opt.step()
            return float(loss.item())
        return "reference", step
    sd = O.make_state_dict(cfg, CH, CH)
    adam = O.AdamState(sd, lr=1e-4)
    return "port", (lambda: O.train_step(hr, sd, cfg, adam, "l2")[0])


def cpu_train_tiles_per_s(which, steps, warmup, threads, budget_s=90.0):
    import torch
    torch.set_num_threads(threads)
    overrides, batch = CPU_WORKLOADS[which]
    kind, step = reference_step_fn(overrides, batch)
    for _ in range(warmup):
        step()
    t0, done = time.perf_counter(), 0
    while done < steps and (done == 0 or time.perf_counter() - t0 < budget_s):
        step()
        done += 1
    dt = time.perf_counter() - t0
    return dict(kind=kind, batch=batch, steps=done, tiles_per_s=batch * done / dt, s_per_step=dt / done)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    steps, warmup = max(1, args.steps), max(1, min(args.warmup, 2))
    full = cpu_train_tiles_per_s("full", steps, warmup, threads, budget_s=60.0)
    small = cpu_train_tiles_per_s("config1", min(steps, 5), 1, threads, budget_s=20.0) if not args.skip_extras else None
    what = "the reference's own sres package (staged copy, oracle/_ref)" if full["kind"] == "reference" else "oracle port of the reference (no copy of the reference found)"
    sample = (f"{full['steps']} timed steps of batch {full['batch']} (of the {BATCH}-tile workload batch), {what}, "
              f"fp32 PyTorch {torch.__version__} CPU, {threads} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": full["tiles_per_s"], "unit": "tiles/s", "n_gpus": args.gpus,
        "steps": full["steps"], "warmup": warmup, "ms_per_step": full["s_per_step"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"RCAN-full (10x20 RCAB, 64 feats, reduction 16) x4 train step, 2-ch 48x48 LR tiles; CPU sample batch {full['batch']}",
                   "tile": TILE, "channels": CH, "scale": SCALE, "batch_per_gpu": BATCH},
        "cpu_baseline": {"value": full["tiles_per_s"], "unit": "tiles/s", "cores": threads, "kind": full["kind"], "sample": sample},
        "e2e": {"value": full["tiles_per_s"], "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if small is not None:
        line["config1"] = {"what": "BASELINE config 1: RCAN-small (4 groups x 4 RCABs, 64 feats) x4 train step, batch 16, CPU",
                           "value": small["tiles_per_s"], "unit": "tiles/s", "ms_per_step": small["s_per_step"] * 1e3,
                           "steps": small["steps"], "kind": small["kind"], "cores": threads}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess():
    """The reference arm in a fresh interpreter (this process has the product's `sres` mirror imported, the reference's
    package has the same name).  Rank 0, N = 1 only."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1",
                              "--skip-extras"], capture_output=True, text=True, timeout=600)
        ref = json.loads(out.stdout.strip().splitlines()[-1])
        return ref["cpu_baseline"]
    except Exception as err:  # the baseline is reporting only: say what happened instead of failing the bench
        return {"value": None, "unit": "tiles/s", "cores": os.cpu_count() or 1, "kind": "unavailable", "sample": f"reference arm failed: {err}"}


# ---------------------------------------------------------------------------------------------------
# BASELINE configs 4 and 5 (extra keys of the main line)
# ---------------------------------------------------------------------------------------------------
def bench_region(trainer, dev, world, rank, reps=3):
    """Config 4 end to end through ModelTrainer.process_image: the (2, 3000, 17280) fp32 region starts in pinned HOST
    memory; tile extraction + NaN-tile drop, lnorm, bicubic down, RCAN-full forward (no grad), de-normalise + stitch, and the
    copy of the stitched images (input / target / interpolated / model of both variables) back to host memory are all
    inside the timed region.  Under torchrun rank 0 copies the region to its GPU and broadcasts it, the tile batches are
    sharded over the ranks, the products are gathered and rank 0 stitches and copies the images out."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from sres.base.util.config import cfg
    from sres.controller.config import TSet
    from sres.data.batch import BatchDataset, synthetic_region
    C_, Y, X = CH, 3000, 17280
    region = torch.from_numpy(synthetic_region(C_, Y, X, seed=12)).pin_memory()
    saved_order, saved_ds = cfg().task.get("tile_order", "reference"), trainer.model_manager._dataset
    cfg().task["tile_order"] = "corrected"
    trainer.model_manager._dataset = BatchDataset(region_source=lambda t: region.numpy())
    trainer.model.eval()
    times, ntiles, bytes_out = [], 0, 0
    try:
        for rep in range(reps + 1):          # rep 0 warms up (workspace, CUDA graph of the inference shape, pinned buffers)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            images, _ = trainer.process_image(TSet.Train, 0, ctime=rep)
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            if rep > 0:
                times.append(float(dt.item()))
            ntiles = int(trainer.get_dataset().timeslice.shape[0])     # tiles that survived the NaN-tile drop
            if rank == 0:   # (under torchrun the images are stitched and copied to the host on rank 0 only)
                img = images[list(images)[0]]["model"]
                assert int(np.isfinite(img[::TILE * SCALE, ::TILE * SCALE]).sum()) == ntiles
                bytes_out = sum(a.nbytes for v in images.values() for a in v.values())
                del img
            del images
    finally:
        cfg().task["tile_order"] = saved_order
        trainer.model_manager._dataset = saved_ds
        trainer.model.train()
    best = min(times)
    mp = C_ * ntiles * (TILE * SCALE) ** 2 / 1e6
    return {"what": "BASELINE config 4: process_image on a synthetic (2, 3000, 17280) region (15 x 90 grid of 192-px tiles, ~20 % land): "
                    "extract, lnorm, bicubic down, RCAN-full forward, denorm + stitch, stitched images copied to host",
            "value": mp / best, "unit": "output MP/s", "seconds": best, "seconds_all": times, "valid_tiles": ntiles, "variables": C_,
            "h2d_bytes": int(region.numel() * 4), "d2h_bytes": int(bytes_out), "n_gpus": world,
            "frac_of_tensor_peak": (C_ * ntiles / C_) / best * flops_per_tile(False) / 1e12 / world / peaks()["tflops_sustained"]}


def bench_x8(dev, world, rank, steps, batch=8):
    """Config 5: RCAN-full x8 (three PixelShuffle(2) stages) on 4-channel 96 x 96 LR tiles -> 768 x 768, one optimizer step
    per step (bicubic down, forward, RMSE, backward, Adam), `batch` tiles per GPU."""
    import torch
    import torch.distributed as dist
    from sres_b200 import nn as snn
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    C4, LR, SC = 4, 96, 8
    torch.manual_seed(4456)
    model = snn.RCAN(nchannels_in=C4, nchannels_out=C4, nfeatures=64, nlayers=WORKLOAD["nlayers"], nblocks=WORKLOAD["nblocks"],
                     cbottleneck=WORKLOAD["cbottleneck"], scale=SC, device=dev)
    group = None
    if world > 1:
        model.enable_data_parallel()
        dist.broadcast(model.engine.flat, src=0)
        model.engine.mark_params_changed()
        group = dist.group.WORLD
    opt = snn.FusedAdam(model, lr=1e-4)
    hr = [synth_hr(batch, C4, LR * SC, 99 + 7 * rank + i).to(dev) for i in range(2)]

    def step(i):
        opt.zero_grad()
        x = snn.bicubic_resize(hr[i % 2], 1.0 / SC)
        loss = snn.loss(model(x.requires_grad_(True)), hr[i % 2], "l2", group)
        loss.backward()
        opt.step()
        return loss

    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        last = step(i)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    Fn, G, R, red = 64, WORKLOAD["nlayers"], WORKLOAD["nblocks"], WORKLOAD["cbottleneck"]
    ups = sum(4 * Fn * Fn * 4 ** i for i in range(3))
    fwd = 2 * 9 * LR * LR * (C4 * Fn + (G * (2 * R + 1) + 1) * Fn * Fn + ups + Fn * C4 * SC * SC) + G * R * 4 * Fn * Fn / red
    tiles_s = world * batch / (ms / 1e3)
    finite = bool(torch.isfinite(last).item())
    del model, opt, hr
    torch.cuda.empty_cache()
    return {"what": f"BASELINE config 5: RCAN-full x8 train step on 4-channel 96x96 LR tiles (768x768 HR), batch {batch} per GPU",
            "value": tiles_s, "unit": "tiles/s", "ms_per_step": ms, "batch_per_gpu": batch, "n_gpus": world, "loss_finite": finite,
            "gflop_per_tile_train": 3 * fwd / 1e9,
            "frac_of_tensor_peak": tiles_s / world * 3 * fwd / 1e12 / peaks()["tflops_sustained"]}


# ---------------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------------
def run_cuda(args):
    sys.path.insert(0, PKG)
    import torch
    import torch.distributed as dist
    from sres_b200 import _lib as L
    from sres_b200 import nn as snn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE {world}; using {world}", file=sys.stderr)
    pk = peaks()
    torch.manual_seed(4456)
    # the public API: the reference's own controller surface (sres.controller.dual_trainer.ModelTrainer)
    from sres.base.util.config import ConfigContext
    from sres.controller.dual_trainer import ModelTrainer
    ConfigContext.set_defaults(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local")
    cc = ConfigContext.activate_global("sres", model="rcan-10-20-64", **{
        "model.cbottleneck": WORKLOAD["cbottleneck"], "task.batch_size": BATCH, "task.lr": 1e-4, "pipeline.gpu": local})
    trainer = ModelTrainer(cc)
    model, opt = trainer.model, trainer.optimizer
    model.train()
    if world > 1:
        dist.broadcast(model.engine.flat, src=0)
        model.engine.mark_params_changed()
    eng = model.engine
    B, S = BATCH, TILE * SCALE
    nbuf = 4
    host = [synth_hr(B, CH, S, 4456 + 17 * rank + i).pin_memory() for i in range(nbuf)]
    resident = [h.to(dev) for h in host]
    step = trainer.train_step   # zero_grad, bicubic down, forward, RMSE, backward, Adam (dual_trainer.py:310-323)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- value: inputs resident in HBM ------------------------------------------------------------
    for i in range(args.warmup):
        step(resident[i % nbuf])
    sync_all()
    # kernels per step: the forward / backward numbers are COUNTED by the library while it enqueued (or captured) them
    # (sres_launch_count, read by the engine around its C calls); + bicubic, loss (partial, final, value, grad), Adam
    per_step_launches = eng.launches_forward(TILE, TILE) + eng.launches_backward() + 1 + 4 + 1
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    captured, hook = {}, None
    if args.dump_outputs and rank == 0:   # keeps the model output of each step (train_step returns only the loss)
        hook = model.register_forward_hook(lambda mod, inp, out: captured.update(prediction=out.detach()))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = step(resident[i % nbuf])
    e1.record()
    sync_all()
    clocks = sampler.stop() if rank == 0 else None
    if hook is not None:
        hook.remove()
        dump_outputs(args.dump_outputs, loss, captured.pop("prediction"), eng)
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * args.steps / (ms_total / 1e3)

    # ---- e2e: host buffers through the public trainer-style call, H2D + loss D2H inside the timed region.
    # ModelTrainer.train_stream takes pinned HOST batches and yields one loss per optimizer step; it issues batch i+1's
    # host-to-device copy on a copy stream before it enqueues step i, so every step's copy is inside the timed region but
    # runs under the previous step's kernels; each loss is read back to a python float before the next step is enqueued.
    for lossv in trainer.train_stream(host[i % nbuf] for i in range(2)):
        lossv.item()
    sync_all()
    e0.record()
    for lossv in trainer.train_stream(host[i % nbuf] for i in range(args.steps)):
        lossv.item()                     # pinned host batch in, python float out
    e1.record()
    sync_all()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t.item()) / 1e3)

    # ---- inference (BASELINE config 4, model part): batched forward without gradients, output megapixels/s ------
    model.eval()
    with torch.no_grad():
        for i in range(3):
            trainer.apply_network(resident[i % nbuf])
        sync_all()
        e0.record()
        for i in range(args.steps):
            trainer.apply_network(resident[i % nbuf])
        e1.record()
        sync_all()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    infer_tiles_s = world * B * args.steps / (float(t.item()) / 1e3)
    model.train()

    # ---- roofline of the dominant kernel, timed live with CUDA events on the launching stream -----------------------
    # The RCAB loop runs its two convolutions as ONE fused launch (conv1 + ReLU -> conv2 + pool partials,
    # sres_conv3x3_pair): 2 x 10.87 GFLOP per launch.  With SRES_CONV_FUSE=0 the single conv1 launch is measured instead.
    import ctypes as C
    rows = B * (TILE + 1) * (TILE + 1)
    nact = 24  # rotate over 24 activation buffers (24 x 19.7 MB >> L2) so the operand is not L2-resident
    acts = [torch.randn(rows, 64, device=dev).bfloat16() for _ in range(nact)]
    midb = torch.empty(rows, 64, device=dev, dtype=torch.bfloat16)
    outb = torch.empty(rows, 64, device=dev, dtype=torch.bfloat16)
    wpack = torch.randn(9 * 64 * 64, device=dev).bfloat16()
    bias = torch.zeros(64, device=dev)
    lib = L.lib()
    lib.sres_conv_pair_flag_bytes.restype = C.c_size_t
    partb = torch.zeros(lib.sres_conv_mtiles(B, TILE, TILE), 2, 4, 64, device=dev)
    flagb = torch.zeros(lib.sres_conv_pair_flag_bytes(B, TILE, TILE) // 4, dtype=torch.int32, device=dev)
    ca = L.ConvArgs()
    ca.wpack_bf16, ca.bias, ca.out_bf16 = wpack.data_ptr(), bias.data_ptr(), midb.data_ptr()
    ca.B, ca.H, ca.W, ca.n_out, ca.epi_flags = B, TILE, TILE, 64, L.EPI_RELU
    cb = L.ConvArgs()
    cb.in_bf16, cb.wpack_bf16, cb.bias, cb.out_bf16, cb.pool_part = midb.data_ptr(), wpack.data_ptr(), bias.data_ptr(), outb.data_ptr(), partb.data_ptr()
    cb.B, cb.H, cb.W, cb.n_out, cb.epi_flags = B, TILE, TILE, 64, L.EPI_POOL
    st = L.cur_stream()
    ca.in_bf16 = acts[0].data_ptr()
    fused = bool(lib.sres_conv_pair_supported(C.byref(ca), C.byref(cb)))

    def launch(i):
        ca.in_bf16 = acts[i % nact].data_ptr()
        if fused:
            return lib.sres_conv3x3_pair(C.byref(ca), C.byref(cb), C.c_void_p(flagb.data_ptr()), st)
        return lib.sres_conv3x3_igemm(C.byref(ca), st)

    reps = 48
    for i in range(8):
        L.check(launch(i), "conv")
    e0.record()
    for i in range(reps):
        launch(i)
    e1.record()
    torch.cuda.synchronize()
    conv_ms = e0.elapsed_time(e1) / reps
    conv_flops = 2.0 * B * TILE * TILE * 64 * 64 * 9 * (2 if fused else 1)
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12
    kernel_name = ("conv3x3_pair_kernel<17,33> (fused RCAB forward pair: 64->64 conv + bias + ReLU -> 64->64 conv + bias + CA pool partials, bf16 out, B=64, 48x48)"
                   if fused else "conv3x3_igemm_kernel<64,false,17> (64->64 conv + bias + ReLU, bf16 out: RCAB conv1, B=64, 48x48)")

    # ---- BASELINE configs 4 and 5 (all ranks take part) ------------------------------------------------
    region = x8 = None
    if not args.skip_extras:
        del acts, outb, midb
        torch.cuda.empty_cache()
        region = bench_region(trainer, dev, world, rank)
        x8 = bench_x8(dev, world, rank, max(3, min(args.steps, 10)))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline: the reference arm on a bounded sample, host cores of this box (N = 1 only) -----
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess()

    # DRAM traffic of the dominant kernel: NOT measured in this run -- read from the committed `ncu --set full` capture of
    # the same kernel and shape (profiles/r02_pair_ncu_metrics.json for the fused pair, profiles/r01_v4_conv_ncu_metrics.json
    # for the single convolution)
    traffic = None
    cap = "r02_pair_ncu_metrics.json" if fused else "r01_v4_conv_ncu_metrics.json"
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", cap)))
        conv = {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "Gbyte": 1e9}
        traffic = sum(float(m[k]["value"].replace(",", "")) * conv[m[k]["unit"]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
    except Exception:
        pass
    step_tflops = value / world * flops_per_tile(True) / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "RCAN-full (10 groups x 20 RCABs, 64 feats, reduction 16) x4 train step: bicubic down, fwd, RMSE, bwd, Adam",
                   "tile": TILE, "channels": CH, "scale": SCALE, "batch_per_gpu": B, "global_batch": B * world,
                   "parallelism": f"dp{world}", "operands": "bf16 tensor-core operands, fp32 accumulate / trunk / grads",
                   "l2": "per-step working set ~12 GB of saved activations >> 126 MB L2; inputs rotate over 4 buffers"},
        "e2e": {"value": e2e_value, "unit": "tiles/s", "h2d_bytes_per_step": B * CH * S * S * 4, "d2h_bytes_per_step": 4},
        "gpu_launches": per_step_launches * args.steps,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": kernel_name, "achieved": achieved, "flops_per_launch": conv_flops,
                     "peak": pk["tflops_burst"], "unit": "TFLOP/s", "frac": achieved / pk["tflops_burst"], "traffic": traffic,
                     "traffic_note": f"from committed capture (ncu --set full, profiles/{cap}), not measured in this run: DRAM bytes per launch; "
                                     + ("algorithmic 59 MB (19.7 in + 19.7 intermediate + 19.7 out): the intermediate and the output are still in L2 when the kernel ends"
                                        if fused else "algorithmic 39.3 MB (19.7 in + 19.7 out): the input is read once, the output is still in L2 when the kernel ends"),
                     "peak_source": pk["src"] + " burst (kernel timed alone)", "us_per_launch": conv_ms * 1e3,
                     "step_tflops_per_gpu": step_tflops, "step_frac_of_sustained": step_tflops / pk["tflops_sustained"]},
        "cpu_baseline": cpu,
        "inference": {"value": infer_tiles_s * (TILE * SCALE) ** 2 / 1e6, "unit": "output MP/s", "tiles_per_s": infer_tiles_s,
                      "what": "bicubic down + RCAN-full forward (no grad) on resident 64-tile batches, all GPUs",
                      "frac_of_tensor_peak": infer_tiles_s / world * flops_per_tile(False) / 1e12 / pk["tflops_sustained"]},
    }
    if region is not None:
        line["infer_region"] = region
        line["x8"] = x8
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="leave out the config-4 / config-5 keys (and config 1 of the reference arm)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss, prediction and parameter / gradient "
                                                          "samples to DIR/*.npy (CUDA arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to the CUDA arm")
    args.warmup = max(args.warmup, 3) if args.impl == "cuda" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
