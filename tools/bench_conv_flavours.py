"""Isolated timing of the four convolution flavours one RCAB runs (forward conv1 / conv2, backward dgrad2 / dgrad1)
on B=64 48x48, same buffers every launch (L2-warm, like consecutive layers of the network)."""
import ctypes as C, os, sys, torch
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "super-resolution-climate_b200"))
from sres_b200 import _lib as L
lib = L.lib(); dev = torch.device("cuda:0")
B, H, W = 64, 48, 48
rows = lib.sres_ptl_rows(B, H, W); nt = lib.sres_conv_mtiles(B, H, W)
xin = (torch.randn(rows, 64, device=dev)).bfloat16()
msk = (torch.randn(rows, 64, device=dev)).bfloat16()
o16 = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
f32 = torch.randn(rows, 64, device=dev)
pool = torch.zeros(nt, 2, 4, 64, device=dev)
w = (torch.randn(64, 64, 3, 3, device=dev) * 0.05)
wpack = torch.empty(9 * 64 * 64, device=dev, dtype=torch.bfloat16)
L.check(lib.sres_pack_conv_weights(L.ptr(w), L.ptr(wpack), 0, 64, 64, 64, 1, 0, L.cur_stream()), "pack")
bias = torch.randn(64, device=dev)
def mk(**kw):
    a = L.ConvArgs(); a.in_bf16 = xin.data_ptr(); a.wpack_bf16 = wpack.data_ptr(); a.B, a.H, a.W = B, H, W; a.n_out = 64
    for k, v in kw.items(): setattr(a, k, v)
    return a
base = {
  "conv1 fwd (bias, relu, bf16 out)": dict(bias=bias.data_ptr(), out_bf16=o16.data_ptr(), epi_flags=L.EPI_RELU),
  "conv2 fwd (bias, pool, bf16 out)": dict(bias=bias.data_ptr(), out_bf16=o16.data_ptr(), epi_flags=L.EPI_POOL, pool_part=pool.data_ptr()),
  "dgrad2    (relu mask, bf16 out) ": dict(out_bf16=o16.data_ptr(), mask_bf16=msk.data_ptr()),
  "dgrad1    (fp32 rmw + dot)      ": dict(out_f32=f32.data_ptr(), resid_f32=f32.data_ptr(), mask_bf16=msk.data_ptr(), epi_flags=4, pool_part=pool.data_ptr()),
  "bf16 out only                   ": dict(bias=bias.data_ptr(), out_bf16=o16.data_ptr()),
}
flav = {k + " specialised": mk(**v) for k, v in base.items()}
st_ = L.cur_stream()
for name, a in flav.items():
    for _ in range(5): L.check(lib.sres_conv3x3_igemm(C.byref(a), st_), name)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(40): lib.sres_conv3x3_igemm(C.byref(a), st_)
    e.record(); torch.cuda.synchronize()
    us = s.elapsed_time(e) / 40 * 1e3
    print(f"{name}  {us:6.1f} us   {2.0*B*H*W*64*64*9/us/1e6:6.0f} TFLOP/s")
