"""Step time and narrow-kernel times of RCAN-full x4 (48 x 48 LR tiles, batch 64) at 2, 4, 8 and 16 image channels.

    python tools/bench_channels.py [--steps 30] [--warmup 5] [--channels 2,4,8,16] [--json OUT]

For each channel count C (C inputs, C targets):
  * the median time of one training step (bicubic down, forward, RMSE, backward, fused Adam) over --steps steps after
    --warmup, with the library's default settings, each step bracketed by CUDA events;
  * in a separate process with SRES_PROFILE=1 (eager launches, no side stream -- tracing slows the host, so these are not
    step times), the per-call time of the four narrow CUDA-core convolutions: "head conv", "head wgrad" (48 x 48 LR
    positions) and "tail dgrad", "tail wgrad" (192 x 192 HR positions).
Each narrow kernel is printed next to its FMA floor: 2 * 9 * C * 64 FLOP per position at the rate the same kernel reaches
at 4 channels, so "x floor" is its time per FLOP relative to the 4-channel run.  The card's name and power limit are read
in the same run.  Nothing is written into the repository (--json writes where it is told).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "super-resolution-climate_b200"))
B, LR, SCALE = 64, 48, 4
KERNELS = {"head conv": LR * LR, "head wgrad": LR * LR, "tail dgrad": (LR * SCALE) ** 2, "tail wgrad": (LR * SCALE) ** 2}


def _model(ch, dev):
    import torch
    from sres_b200 import nn as snn
    torch.manual_seed(4456)
    m = snn.RCAN(nchannels_in=ch, nchannels_out=ch, nfeatures=64, nlayers=10, nblocks=20, cbottleneck=16, scale=SCALE,
                 device=dev)
    opt = snn.FusedAdam(m, lr=1e-4)
    g = torch.Generator(device=dev).manual_seed(99 + ch)
    hr = [torch.randn(B, ch, LR * SCALE, LR * SCALE, device=dev, generator=g) for _ in range(2)]

    def step(i):
        opt.zero_grad()
        loss = snn.loss(m(snn.bicubic_resize(hr[i % 2], 1.0 / SCALE).requires_grad_(True)), hr[i % 2], "l2")
        loss.backward()
        opt.step()
        return loss
    return step


def time_steps(ch, steps, warmup):
    import torch
    dev = torch.device("cuda:0")
    step = _model(ch, dev)
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i, (e0, e1) in enumerate(ev):
        e0.record()
        loss = step(i)
        e1.record()
    torch.cuda.synchronize()
    assert torch.isfinite(loss).item()
    ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    return statistics.median(ms), min(ms), max(ms)


def profile(ch):
    """Runs in a child process with SRES_PROFILE=1: per-category {name: (calls, total ms)} of the last of 4 steps."""
    import torch
    from sres_b200 import _lib as L
    dev = torch.device("cuda:0")
    step = _model(ch, dev)
    buf = C.create_string_buffer(16384)
    for i in range(4):
        step(i)
        torch.cuda.synchronize()
        L.check(L.lib().sres_profile_report(buf, C.c_size_t(len(buf))), "sres_profile_report")
    out = {}
    for line in buf.value.decode().splitlines():
        for k in KERNELS:
            if line.startswith(k) and " n=" in line:
                n = int(line.split("n=")[1].split()[0])
                ms = float(line.split("n=")[1].split()[1])
                out[k] = (n, ms)
    return out


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return q.stdout.strip() or name
    except (OSError, subprocess.SubprocessError):
        return f"{name}, power limit not readable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--channels", default="2,4,8,16")
    ap.add_argument("--json", default=None)
    ap.add_argument("--profile-child", type=int, default=0, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.profile_child:
        print(json.dumps(profile(a.profile_child)))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_channels.py: needs a CUDA device")
    if a.steps < 20:
        raise SystemExit("--steps: at least 20")
    chans = [int(c) for c in a.channels.split(",")]
    dev_line = card()
    print(f"device: {dev_line}")
    print(f"RCAN-full x4 (10 groups x 20 RCABs, reduction 16), {LR}x{LR} LR tiles, batch {B}; median of {a.steps} steps "
          f"after {a.warmup}")
    res = {}
    for ch in chans:
        med, lo, hi = time_steps(ch, a.steps, a.warmup)
        env = dict(os.environ, SRES_PROFILE="1", SRES_CUDA_GRAPHS="0", SRES_SIDE_STREAM="0")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--profile-child", str(ch)], env=env,
                           capture_output=True, text=True, check=True)
        prof = json.loads(r.stdout.strip().splitlines()[-1])
        res[ch] = dict(step_ms_median=med, step_ms_min=lo, step_ms_max=hi,
                       kernels={k: dict(calls=v[0], ms_per_step=v[1]) for k, v in prof.items()})
        print(f"  C = {ch:2d}: step {med:8.3f} ms (min {lo:.3f}, max {hi:.3f})")
    print()
    ref = 4 if 4 in res else None
    print(f"{'kernel':<12s} {'C':>3s} {'ms/step':>9s} {'GFLOP':>8s} {'TFLOP/s':>8s} {'floor ms':>9s} {'x floor':>8s}")
    for k, pos in KERNELS.items():
        for ch in chans:
            kk = res[ch]["kernels"].get(k)
            if kk is None:
                continue
            gflop = 2 * 9 * ch * 64 * B * pos / 1e9
            ms = kk["ms_per_step"]
            rate = gflop / ms   # GFLOP per ms = TFLOP/s
            floor = None
            if ref is not None and k in res[ref]["kernels"]:
                rate4 = (2 * 9 * ref * 64 * B * pos / 1e9) / res[ref]["kernels"][k]["ms_per_step"]
                floor = gflop / rate4
            kk.update(gflop=gflop, tflops=rate, floor_ms=floor)
            fl = f"{floor:9.3f} {ms / floor:8.2f}" if floor else f"{'-':>9s} {'-':>8s}"
            print(f"{k:<12s} {ch:3d} {ms:9.3f} {gflop:8.2f} {rate:8.1f} {fl}")
    out = dict(device=dev_line, batch=B, lr_tile=LR, scale=SCALE, steps=a.steps, warmup=a.warmup, results=res)
    print(json.dumps(out))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
