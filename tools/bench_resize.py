"""Resize kernels per interpolation mode, and the training step with each downsample mode.

    python tools/bench_resize.py [--channels 2] [--launches 200] [--steps 30] [--warmup 5] [--rounds 3] [--json OUT]

  * Per mode (nearest, nearest-exact, bilinear, bicubic, area) the training-shape downsample, 64 x C x 192^2 -> 48^2
    (x4), and the evaluation-shape upsample, 64 x C x 48^2 -> 192^2, through `sres_resize`.  Kernel time is the device
    duration torch.profiler records for each launch (median over --launches eager launches, in a child process: tracing
    slows the host, so nothing else is timed there).  The launches rotate over input / output buffers that together hold
    more than 4x the 126 MB L2, so every launch reads its input from HBM.  GB/s counts the input tensor read once plus the
    output tensor written once (nearest and bilinear downsamples touch fewer input sectors than that) against the
    6545 GB/s HBM peak measured on this pool (DESIGN.md section 3).  Each mode's output at the timed shape is compared
    with F.interpolate on the GPU first.
  * The median training step (RCAN-full x4, 48 x 48 LR tiles, batch 64, C channels; down-sampling, forward, RMSE,
    backward, fused Adam), each step bracketed by CUDA events like tools/bench_channels.py, with the down-sampling of
    downsample_mode = cubic (the `bicubic_resize` the default configuration runs), linear and area.  The modes take turns
    for --rounds rounds of --steps steps on one model, so drift over the run falls on all of them alike.
The card's name and power limit are read in the same run.  Nothing is written into the repository (--json writes where
it is told).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "super-resolution-climate_b200"))
sys.path.insert(0, HERE)
from bench_channels import B, LR, SCALE, card  # noqa: E402

MODES = ["nearest", "nearest-exact", "bilinear", "bicubic", "area"]
STEP_MODES = {"cubic": "bicubic", "linear": "bilinear", "area": "area"}   # task.downsample_mode -> F.interpolate mode
HBM_GBS = 6545.0
L2_BYTES = 126 << 20


def _shapes(ch):
    hr, lr = LR * SCALE, LR
    return {"down": ((B, ch, hr, hr), (B, ch, lr, lr), 1.0 / SCALE), "up": ((B, ch, lr, lr), (B, ch, hr, hr), float(SCALE))}


def kernel_times(ch, launches):
    """Child process: {direction: {mode: dict(us, bytes, max_abs_diff)}}."""
    import torch
    import torch.nn.functional as F
    from sres_b200 import _lib as L
    from sres_b200 import nn as snn
    dev = torch.device("cuda:0")
    lib = L.lib()
    out = {}
    for direction, (ishape, oshape, sf) in _shapes(ch).items():
        nin, nout = math.prod(ishape), math.prod(oshape)
        nbytes = 4 * (nin + nout)
        nbuf = max(2, -(-4 * L2_BYTES // nbytes))
        g = torch.Generator(device=dev).manual_seed(7)
        ins = [torch.randn(ishape, device=dev, generator=g) for _ in range(nbuf)]
        outs = [torch.empty(oshape, device=dev) for _ in range(nbuf)]
        Hi, Wi, Ho, Wo = ishape[2], ishape[3], oshape[2], oshape[3]
        res = {}
        for mode in MODES:
            ref = F.interpolate(ins[0], scale_factor=sf, mode=mode)
            diff = (snn.resize(ins[0], sf, mode) - ref).abs().max().item()

            def launch(i):
                L.check(lib.sres_resize(L.ptr(ins[i % nbuf]), L.ptr(outs[i % nbuf]), B * ch, Hi, Wi, Ho, Wo, 1.0 / sf,
                                        1.0 / sf, L.RESIZE_MODES[mode], L.cur_stream()), "sres_resize")
            for i in range(2 * nbuf):
                launch(i)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for i in range(launches):
                    launch(i)
                torch.cuda.synchronize()
            durs = [e.time_range.elapsed_us() for e in prof.events()
                    if e.device_type == torch.autograd.DeviceType.CUDA and "resize_kernel" in e.name]
            if len(durs) != launches:
                raise SystemExit(f"bench_resize.py: the profiler recorded {len(durs)} resize kernels for {launches} launches")
            res[mode] = dict(us=statistics.median(durs), us_min=min(durs), bytes=nbytes, max_abs_diff=diff)
        out[direction] = dict(input=list(ishape), output=list(oshape), buffers=nbuf, modes=res)
        del ins, outs
        torch.cuda.empty_cache()
    return out


def step_times(ch, steps, warmup, rounds):
    import torch
    from sres_b200 import nn as snn
    dev = torch.device("cuda:0")
    torch.manual_seed(4456)
    m = snn.RCAN(nchannels_in=ch, nchannels_out=ch, nfeatures=64, nlayers=10, nblocks=20, cbottleneck=16, scale=SCALE,
                 device=dev)
    opt = snn.FusedAdam(m, lr=1e-4)
    g = torch.Generator(device=dev).manual_seed(99 + ch)
    hr = [torch.randn(B, ch, LR * SCALE, LR * SCALE, device=dev, generator=g) for _ in range(2)]

    def step(i, mode):
        opt.zero_grad()
        x = snn.bicubic_resize(hr[i % 2], 1.0 / SCALE) if mode == "bicubic" else snn.resize(hr[i % 2], 1.0 / SCALE, mode)
        loss = snn.loss(m(x.requires_grad_(True)), hr[i % 2], "l2")
        loss.backward()
        opt.step()
        return loss

    for name, mode in STEP_MODES.items():
        for i in range(warmup):
            step(i, mode)
    torch.cuda.synchronize()
    ms = {name: [] for name in STEP_MODES}
    per_round = {name: [] for name in STEP_MODES}
    for _ in range(rounds):
        for name, mode in STEP_MODES.items():
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for i, (e0, e1) in enumerate(ev):
                e0.record()
                loss = step(i, mode)
                e1.record()
            torch.cuda.synchronize()
            assert torch.isfinite(loss).item()
            t = [e0.elapsed_time(e1) for e0, e1 in ev]
            ms[name] += t
            per_round[name].append(statistics.median(t))
    return {name: dict(step_ms_median=statistics.median(v), step_ms_min=min(v), step_ms_max=max(v),
                       round_medians=per_round[name]) for name, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=2)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", default=None)
    ap.add_argument("--kernel-child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.kernel_child:
        print(json.dumps(kernel_times(a.channels, a.launches)))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_resize.py: needs a CUDA device")
    if a.steps < 20 or a.launches < 50 or a.rounds < 1:
        raise SystemExit("--steps: at least 20; --launches: at least 50; --rounds: at least 1")
    ch = a.channels
    dev_line = card()
    print(f"device: {dev_line}")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--kernel-child", "--channels", str(ch),
                        "--launches", str(a.launches)], capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit(f"bench_resize.py: kernel timing failed:\n{r.stdout}\n{r.stderr}")
    kern = json.loads(r.stdout.strip().splitlines()[-1])
    for direction, d in kern.items():
        print(f"{direction}: {tuple(d['input'])} -> {tuple(d['output'])}, {d['buffers']} buffer pairs in rotation, median "
              f"kernel time of {a.launches} launches (torch.profiler)")
        print(f"  {'mode':<14s} {'us':>8s} {'min us':>8s} {'MB':>7s} {'GB/s':>7s} {'% HBM':>6s} {'max |d| vs F.interpolate':>26s}")
        for mode, k in d["modes"].items():
            gbs = k["bytes"] / (k["us"] * 1e3)
            k.update(gbs=gbs, hbm_frac=gbs / HBM_GBS)
            print(f"  {mode:<14s} {k['us']:8.2f} {k['us_min']:8.2f} {k['bytes'] / 1e6:7.2f} {gbs:7.0f} {100 * gbs / HBM_GBS:6.1f} "
                  f"{k['max_abs_diff']:26.2e}")
    print(f"training step, RCAN-full x4 (10 groups x 20 RCABs, reduction 16), {LR}x{LR} LR tiles, batch {B}, {ch} channels; "
          f"{a.rounds} rounds x {a.steps} steps per mode after {a.warmup}")
    steps = step_times(ch, a.steps, a.warmup, a.rounds)
    for name, s in steps.items():
        rounds = " / ".join(f"{v:.2f}" for v in s["round_medians"])
        print(f"  downsample_mode {name:<6s}: median {s['step_ms_median']:7.3f} ms (min {s['step_ms_min']:.3f}, "
              f"max {s['step_ms_max']:.3f}; round medians {rounds})")
    out = dict(device=dev_line, batch=B, lr_tile=LR, scale=SCALE, channels=ch, hbm_gbs=HBM_GBS, kernels=kern, steps=steps)
    print(json.dumps(out))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
