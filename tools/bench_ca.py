"""Microbenchmark of ca_apply_fwd / ca_bwd on B=64 48x48 with rotating (cold) and fixed (L2-hot) buffers."""
import ctypes as C, os, sys, torch
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "super-resolution-climate_b200"))
from sres_b200 import _lib as L
lib = L.lib(); dev = torch.device("cuda:0")
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
H, W, hid = 48, 48, 4
rows = B * 49 * 49
nt = lib.sres_conv_mtiles(B, H, W)
NB = 12
t2 = [torch.randn(rows, 64, device=dev).bfloat16() for _ in range(NB)]
x = [torch.randn(rows, 64, device=dev) for _ in range(NB)]
xb = [torch.empty(rows, 64, device=dev, dtype=torch.bfloat16) for _ in range(NB)]
pool = torch.randn(nt, 2, 4, 64, device=dev)
w1, b1, w2, b2 = torch.randn(hid, 64, device=dev), torch.randn(hid, device=dev), torch.randn(64, hid, device=dev), torch.randn(64, device=dev)
mean, sv, ds = torch.empty(B, 64, device=dev), torch.empty(B, 64, device=dev), torch.empty(B, 64, device=dev)
bpi = lib.sres_ca_blocks_per_image(B, H, W)
dsp = torch.empty(B * bpi * 64, device=dev)
st = L.cur_stream()
def fwd(i): return lib.sres_ca_apply_fwd(L.ptr(t2[i]), L.ptr(pool), None, L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), hid, L.ptr(x[i]), L.ptr(x[i]), L.ptr(xb[i]), L.ptr(mean), L.ptr(sv), B, H, W, st)
def bwd(i): return lib.sres_ca_bwd(L.ptr(x[i]), L.ptr(t2[i]), L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), hid, L.ptr(mean), L.ptr(dsp), L.ptr(xb[i]), L.ptr(ds), B, H, W, st)
lib.sres_ca_bwd_apply.restype = C.c_int
def bwd_apply(i): return lib.sres_ca_bwd_apply(L.ptr(x[i]), L.ptr(pool), L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), hid, L.ptr(mean), L.ptr(xb[i]), L.ptr(ds), B, H, W, st)
def timeit(fn, rot, n=48):
    for i in range(6): L.check(fn(i % NB if rot else 0), "k")
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n): fn(i % NB if rot else 0)
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3
print(f"bpi={bpi}  ca_apply_fwd: cold {timeit(fwd, True):.1f} us, hot {timeit(fwd, False):.1f} us   (118 MB at B=64); B={B}, {118e6*B/64/timeit(fwd, False)/1e6:.2f} TB/s hot")
print(f"bpi={bpi}  ca_bwd (2 kernels): cold {timeit(bwd, True):.1f} us, hot {timeit(bwd, False):.1f} us   (2 x 59 MB)")
print(f"bpi={bpi}  ca_bwd_apply (fused-dot path, in-network kernel): cold {timeit(bwd_apply, True):.1f} us, hot {timeit(bwd_apply, False):.1f} us   (59 MB at B=64)")
