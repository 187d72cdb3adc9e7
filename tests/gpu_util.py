"""Helpers for the GPU parity tests: padded-tile-layout conversion and ctypes plumbing."""
import ctypes as C

import torch

from sres_b200 import _lib as L


def to_ptl(x_nchw: torch.Tensor, dtype) -> torch.Tensor:
    B, Cc, H, W = x_nchw.shape
    out = torch.zeros(B, H + 1, W + 1, Cc, device=x_nchw.device, dtype=dtype)
    out[:, :H, :W, :] = x_nchw.permute(0, 2, 3, 1).to(dtype)
    return out.reshape(B * (H + 1) * (W + 1), Cc).contiguous()


def from_ptl(p: torch.Tensor, B, H, W) -> torch.Tensor:
    return p.reshape(B, H + 1, W + 1, p.shape[-1])[:, :H, :W, :].permute(0, 3, 1, 2).float().contiguous()


def pads_are_zero(p: torch.Tensor, B, H, W) -> bool:
    full = p.reshape(B, H + 1, W + 1, p.shape[-1]).float()
    return bool((full[:, H] == 0).all() and (full[:, :, W] == 0).all())


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.bfloat16().float()


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


def conv3x3_wgrad_ref(x: torch.Tensor, dy: torch.Tensor):
    """Weight gradient of a 3x3, padding-1 convolution in float64 as nine shifted reductions,
    dW[o,i,ky,kx] = sum_{b,y,x} dy[b,o,y,x] * xpad[b,i,y+ky,x+kx], and the same reduction over |x|, |dy| (the scale
    against which the fp32 rounding of each element is judged).  x (B,Ci,H,W), dy (B,Co,H,W) -> two (Co,Ci,3,3)."""
    H, W = dy.shape[2:]
    xp = torch.nn.functional.pad(x.double(), (1, 1, 1, 1))
    d = dy.double()
    dw = torch.empty(dy.shape[1], x.shape[1], 3, 3, dtype=torch.float64, device=dy.device)
    A = torch.empty_like(dw)
    for ky in range(3):
        for kx in range(3):
            xs = xp[:, :, ky:ky + H, kx:kx + W]
            dw[:, :, ky, kx] = torch.tensordot(d, xs, dims=([0, 2, 3], [0, 2, 3]))
            A[:, :, ky, kx] = torch.tensordot(d.abs(), xs.abs(), dims=([0, 2, 3], [0, 2, 3]))
    return dw, A


def check_grad(name, got, ref, A, rel_bound, elem=2.0 ** -12):
    """Compare a kernel's gradient tensor with its float64 reference: rel-L2 below `rel_bound` and every element within
    `elem` * A (A = the reduction over absolute values).  Prints both measured numbers (visible with pytest -s)."""
    d = (got.double() - ref.double()).abs()
    rel = (d.norm() / (ref.double().norm() + 1e-300)).item()
    worst = (d / A.double().clamp_min(1e-300)).max().item()
    print(f"  {name:<44s} rel-L2 {rel:.2e} (bound {rel_bound:.0e})   max|err|/A {worst:.2e}")
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    assert rel < rel_bound, f"{name}: rel-L2 {rel:.3e} >= {rel_bound:.0e}"
    assert bool((d <= elem * A.double()).all()), f"{name}: worst element |err|/A = {worst:.3e} > {elem:.3e}"
    return rel


def pack(lib, w: torch.Tensor, mode: int, n_rows=64, stride=1, offset=0) -> torch.Tensor:
    out = torch.empty(9 * n_rows * 64, device=w.device, dtype=torch.bfloat16)
    _KEEP.append(w)
    L.check(lib.sres_pack_conv_weights(L.ptr(w), L.ptr(out), mode, n_rows, w.shape[1], w.shape[0], stride, offset, L.cur_stream()), "pack")
    return out


_KEEP = []  # tensors whose device pointers were handed to the C ABI stay alive until the test session ends


def ptr(t):
    """Device pointer of `t` (None -> NULL) that keeps `t` alive: `L.ptr(x.to(dev))` would free the
    temporary before the kernel runs and let the caching allocator hand its memory to the next tensor."""
    if t is not None:
        _KEEP.append(t)
        if len(_KEEP) > 4096:
            torch.cuda.synchronize()
            del _KEEP[:2048]
    return L.ptr(t)


def conv_args(**kw) -> L.ConvArgs:
    a = L.ConvArgs()
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            _KEEP.append(v)
            v = v.data_ptr()
        setattr(a, k, v)
    return a


def run_conv(lib, a: L.ConvArgs):
    L.check(lib.sres_conv3x3_igemm(C.byref(a), L.cur_stream()), "sres_conv3x3_igemm")
    torch.cuda.synchronize()
