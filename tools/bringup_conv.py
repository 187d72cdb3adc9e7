"""GPU bring-up check of the tcgen05 conv kernel against torch (fp32 math on bf16-rounded operands).
Run on a B200:  python tools/bringup_conv.py --B 2 --H 48 --W 48 [--debug-flags 1]
"""
import argparse
import ctypes as C
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "super-resolution-climate_b200"))
from sres_b200 import _lib as L  # noqa: E402


def to_ptl(x_nchw, dtype):
    B, Cc, H, W = x_nchw.shape
    out = torch.zeros(B, H + 1, W + 1, Cc, device=x_nchw.device, dtype=dtype)
    out[:, :H, :W, :] = x_nchw.permute(0, 2, 3, 1).to(dtype)
    return out.reshape(B * (H + 1) * (W + 1), Cc).contiguous()


def from_ptl(p, B, H, W):
    Cc = p.shape[-1]
    return p.reshape(B, H + 1, W + 1, Cc)[:, :H, :W, :].permute(0, 3, 1, 2).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=2)
    ap.add_argument("--H", type=int, default=48)
    ap.add_argument("--W", type=int, default=48)
    ap.add_argument("--nout", type=int, default=64)
    ap.add_argument("--debug-flags", type=int, default=0)
    ap.add_argument("--mode", default="fwd", choices=["fwd", "dgrad", "relu_pool", "shuffle", "resid"])
    ap.add_argument("--iters", type=int, default=0)
    ap.add_argument("--bf16-only", action="store_true")
    ap.add_argument("--timeline", action="store_true")
    ap.add_argument("--relu", action="store_true", help="fwd mode: fuse ReLU (with --bf16-only this is the RCAB conv1 flavour)")
    a = ap.parse_args()
    torch.manual_seed(0)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    lib = L.lib()
    B, H, W = a.B, a.H, a.W
    x = torch.randn(B, 64, H, W, device=dev).bfloat16().float()
    cout = 64 if a.nout == 64 else 2
    w = (torch.randn(cout, 64, 3, 3, device=dev) * 0.05).bfloat16().float()
    bias = torch.randn(cout, device=dev)
    xp = to_ptl(x, torch.bfloat16)
    rows = xp.shape[0]
    wpack = torch.empty(9 * a.nout * 64, device=dev, dtype=torch.bfloat16)
    pmode = 1 if a.mode == "dgrad" else 0
    L.check(lib.sres_pack_conv_weights(L.ptr(w), L.ptr(wpack), pmode, a.nout, 64, cout, 1, 0, L.cur_stream()), "pack")
    args = L.ConvArgs()
    args.in_bf16 = xp.data_ptr()
    args.wpack_bf16 = wpack.data_ptr()
    bias_pad = torch.zeros(a.nout, device=dev)
    bias_pad[:cout] = bias
    args.bias = bias_pad.data_ptr()
    args.B, args.H, args.W = B, H, W
    args.n_out = a.nout
    args.debug_flags = a.debug_flags
    out_f32 = torch.full((rows, 64), float("nan"), device=dev)
    out_bf16 = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
    ntiles = lib.sres_conv_mtiles(B, H, W)
    pool = torch.full((ntiles, 2, 4, 64), float("nan"), device=dev)
    ref = None
    if a.nout == 16:
        out_nchw = torch.full((B, cout, H, W), float("nan"), device=dev)
        args.out_nchw = out_nchw.data_ptr()
        args.c_real = cout
        ref = F.conv2d(x, w, bias, padding=1)
    elif a.mode == "fwd":
        args.out_f32 = out_f32.data_ptr()
        args.out_bf16 = out_bf16.data_ptr()
        if a.bf16_only:
            args.out_f32 = None
        ref = F.conv2d(x, w, bias, padding=1)
        if a.relu:
            args.epi_flags = L.EPI_RELU
            ref = F.relu(ref)
    elif a.mode == "dgrad":
        args.out_f32 = out_f32.data_ptr()
        args.bias = None
        ref = F.conv_transpose2d(x, w, None, padding=1)  # = grad_input of conv2d(.., w) for grad_output x
    elif a.mode == "relu_pool":
        args.out_f32 = out_f32.data_ptr()
        args.epi_flags = L.EPI_RELU | L.EPI_POOL
        args.pool_part = pool.data_ptr()
        ref = F.relu(F.conv2d(x, w, bias, padding=1))
    elif a.mode == "resid":
        res = torch.randn(B, 64, H, W, device=dev)
        out_f32 = to_ptl(res, torch.float32)
        args.out_f32 = out_f32.data_ptr()
        args.resid_f32 = out_f32.data_ptr()
        ref = F.conv2d(x, w, bias, padding=1) + res
    elif a.mode == "shuffle":
        rows2 = lib.sres_ptl_rows(B, 2 * H, 2 * W)
        out_bf16 = torch.full((rows2, 64), float("nan"), device=dev, dtype=torch.bfloat16)
        w4 = (torch.randn(256, 64, 3, 3, device=dev) * 0.05).bfloat16().float()
        b4 = torch.randn(256, device=dev)
        ref = F.pixel_shuffle(F.conv2d(x, w4, b4, padding=1), 2)
        for i in range(2):
            for j in range(2):
                L.check(lib.sres_pack_conv_weights(L.ptr(w4), L.ptr(wpack), 0, 64, 64, 256, 4, 2 * i + j, L.cur_stream()), "pack")
                bsub = b4[2 * i + j::4].contiguous()
                args.bias = bsub.data_ptr()
                args.out_bf16 = out_bf16.data_ptr()
                args.map_mode = L.MAP_SHUFFLE
                args.sub_i, args.sub_j = i, j
                L.check(lib.sres_conv3x3_igemm(C.byref(args), L.cur_stream()), "conv")
                torch.cuda.synchronize()
        got = from_ptl(out_bf16, B, 2 * H, 2 * W)
        full = out_bf16.reshape(B, 2 * H + 1, 2 * W + 1, 64).float()
        print("pad row max", full[:, 2 * H].abs().max().item(), "pad col max", full[:, :, 2 * W].abs().max().item())
        err = (got - ref).abs().max().item()
        rel = ((got - ref).norm() / ref.norm()).item()
        print(f"RESULT mode=shuffle B={B} H={H} W={W} max_abs_err={err:.4e} rel_l2={rel:.4e}")
        return

    L.check(lib.sres_conv3x3_igemm(C.byref(args), L.cur_stream()), "conv")
    torch.cuda.synchronize()
    if a.nout == 16:
        got = out_nchw
    else:
        src = out_bf16 if (a.mode == "fwd" and a.bf16_only) else out_f32
        got = from_ptl(src, B, H, W)
        full = src.reshape(B, H + 1, W + 1, 64).float()
        print("pad row max", full[:, H].abs().max().item(), "pad col max", full[:, :, W].abs().max().item())
    err = (got - ref).abs().max().item()
    rel = ((got - ref).norm() / ref.norm()).item()
    print(f"RESULT mode={a.mode} nout={a.nout} dbg={a.debug_flags} B={B} H={H} W={W} max_abs_err={err:.4e} rel_l2={rel:.4e} nan={torch.isnan(got).sum().item()}")
    if a.mode == "fwd" and a.nout == 64:
        gb = from_ptl(out_bf16, B, H, W)
        print("bf16 out rel_l2", ((gb - ref).norm() / ref.norm()).item())
    if a.mode == "relu_pool":
        RP = (H + 1) * (W + 1)
        sums = torch.zeros(B, 64, device=dev)
        for t in range(ntiles):
            b0 = (t * 128) // RP
            for seg in range(2):
                if b0 + seg < B:
                    sums[b0 + seg] += pool[t, seg].sum(0)
        rs = ref.sum(dim=(2, 3))
        print("pool rel err", ((sums - rs).norm() / rs.norm()).item(), "nan", torch.isnan(pool).sum().item())
    if a.iters:
        st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            lib.sres_conv3x3_igemm(C.byref(args), L.cur_stream())
        st.record()
        for _ in range(a.iters):
            lib.sres_conv3x3_igemm(C.byref(args), L.cur_stream())
        en.record()
        torch.cuda.synchronize()
        ms = st.elapsed_time(en) / a.iters
        fl = 2.0 * B * H * W * 64 * (64 if a.nout == 64 else 16) * 9
        print(f"TIMING {ms*1000:.1f} us/conv  {fl/ms/1e9:.1f} TFLOP/s (useful)")
    if a.timeline:
        tl = torch.zeros(148 * 16, dtype=torch.int64, device=dev)
        args.debug_timeline = tl.data_ptr()
        for _ in range(3):
            lib.sres_conv3x3_igemm(C.byref(args), L.cur_stream())
        torch.cuda.synchronize()
        t = tl.cpu().reshape(148, 16).double()
        g0 = t[:, 10].min()
        names = {1: "setup done", 3: "weights landed", 4: "first A tile landed", 6: "first accumulator ready", 5: "last MMA issued",
                 7: "last accumulator ready", 8: "last store issued", 9: "stores drained", 12: "exit"}
        print("per-CTA timeline, cycles since CTA entry (min / median / max over CTAs):")
        for i in (1, 3, 4, 6, 5, 7, 8, 9, 12):
            sel = t[:, i] != 0   # CTAs without a tile stamp nothing
            d = (t[:, i] - t[:, 0])[sel]
            print(f"  {names[i]:26s} {d.min():9.0f} {d.median():9.0f} {d.max():9.0f}")
        for i, nm in ((13, "epilogue warp idle (waits for MMA)"), (14, "MMA warp waits for epilogue"), (15, "MMA warp waits for TMA")):
            d = t[:, i]
            print(f"  total cycles: {nm:36s} {d.min():9.0f} {d.median():9.0f} {d.max():9.0f}")
        st = t[:, 10] - g0; en = t[:, 11] - g0
        print(f"globaltimer ns: CTA start min/med/max {st.min():.0f}/{st.median():.0f}/{st.max():.0f}  end {en.min():.0f}/{en.median():.0f}/{en.max():.0f}")


if __name__ == "__main__":
    main()
