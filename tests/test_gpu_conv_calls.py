"""Tensor-core convolution calls (conv_igemm.cu, conv_pair.cu, conv_n192.cu) against float64 references, one call of
rcan_net.cu at a time, built with the same sres_conv_args fields and run at the shapes the training step runs them at.

These kernels run in every forward pass and every input gradient.  A wrong row, column, tile, sub-pixel or epilogue
operand would spread into every activation and gradient after it, and a whole-tensor norm at toy shapes can miss it.  So
every output here is compared element by element with plain PyTorch in float64, computed from the operands the kernel
reads (bf16 where it reads bf16), and two numbers are printed per tensor (visible with `pytest -s`):

    rel-L2      ||got - ref|| / ||ref||   (bf16 outputs: against the bf16 rounding of ref, so one flipped rounding shows)
    max|err|/A  worst element error over A = the same sum over |operands| (+ |bias| + |addends|), with its
                (image, y, x, channel) so that a failure points at a tile

and each element must satisfy |got - ref| <= 2^-12 A (fp32 outputs) or 2^-8 |ref| + 2^-12 A (bf16 outputs).  Products
of bf16 operands are exact in fp32, so only the fp32 summation order separates a correct kernel from the reference.
Padding rows must be exactly 0, outputs are prefilled with NaN, direct-store outputs have a NaN guard region behind
them, fp32 addends carry NaN in their padding rows (the kernel must zero them, not add them), every call runs twice and
must be bit-identical, and a pair launch must leave its flag buffer all zero.

Shapes: the x4 bench (B = 64, body 48 x 48: 1201 tiles, about 8 per CTA, the last one half full), the x8 bench (body
8 x 96 x 96, upsampler stages at 96 / 192 / 384 and the tail at 768, the last two at B = 2), x3 (one f = 3 stage), and two
edges: 5 x 10 x 11 ((H+1)(W+1) = 132: almost every tile straddles two images) and 37 x 7 x 9 (an image smaller than one
tile: the network then uses no POOL / DOT partials and no pair).
"""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gpu_util
from gpu_util import conv_args, pack, ptr, to_ptl

TILE = 128          # rows per M tile (sres_conv_tile_rows)
GUARD = 256         # NaN rows behind every output buffer
NAN = float("nan")
HID = 4             # channel-attention hidden units of RCAN-full (reduction 16)

# rel-L2 bounds: about 10x the largest value measured on a B200 (NVIDIA B200, 1000 W power limit) over the cases below;
# there every element stayed within 3.5e-7 A (fp32 outputs, 2^-12 = 2.4e-4 allowed), and the file ran in 5 s
REL_F32 = 6e-6      # fp32 outputs: measured <= 5.5e-7 (tail conv <= 1.7e-7)
REL_BF16 = 1e-3     # bf16 outputs, against the bf16 rounding of the fp64 reference: measured <= 1.05e-4
REL_SUM = 6e-6      # per-image sums from the POOL / DOT partials, save_mean, save_s: measured <= 5.5e-7


# ---------------------------------------------------------------------------------------------------------------------
# references and layouts (checked on the CPU by test_reference_helpers_cpu)
# ---------------------------------------------------------------------------------------------------------------------
def conv_ref(x, w, bias=None):
    """3x3, padding-1 convolution in float64 as nine shifted tensordots over the zero-padded input, and the same sum over
    |x| |w| + |bias| (the scale A against which the fp32 rounding of each element is judged).
    x (B,Ci,H,W), w (Co,Ci,3,3) -> two (B,Co,H,W)."""
    B, _, H, W = x.shape
    xp = F.pad(x.double(), (1, 1, 1, 1))
    wd = w.double()
    y = torch.zeros(B, H, W, w.shape[0], dtype=torch.float64, device=x.device)
    A = torch.zeros_like(y)
    for ky in range(3):
        for kx in range(3):
            xs = xp[:, :, ky:ky + H, kx:kx + W]
            y += torch.tensordot(xs, wd[:, :, ky, kx], dims=([1], [1]))
            A += torch.tensordot(xs.abs(), wd[:, :, ky, kx].abs(), dims=([1], [1]))
    if bias is not None:
        y += bias.double()
        A += bias.double().abs()
    return y.permute(0, 3, 1, 2), A.permute(0, 3, 1, 2)


def dgrad_w(w):
    """Weights of the input gradient as a forward convolution: transposed and flipped (conv_transpose2d's)."""
    return w.transpose(0, 1).flip(2, 3)


def ptl_valid(p, B, H, W):
    """(B,H,W,C) view of the valid positions of a PTL buffer."""
    return p.reshape(B, H + 1, W + 1, -1)[:, :H, :W]


def ptl_nchw(p, B, H, W):
    return ptl_valid(p, B, H, W).permute(0, 3, 1, 2)


def unshuffle_ptl(x, f, dtype):
    """PixelUnshuffle layout (SRES_MAP_UNSHUFFLE, sres_rcan_workspace_bytes): x (B,C,fH,fW) as f*f PTL sub-grids of
    (B,H,W), sub-grid (y % f) * f + (x % f) holding position (b, y / f, x / f)."""
    u = F.pixel_unshuffle(x, f)
    return torch.cat([to_ptl(u[:, s::f * f], dtype) for s in range(f * f)])


def from_unshuffle_ptl(p, B, H, W, f):
    """Inverse of unshuffle_ptl: f*f sub-grids of (B,H,W) -> (B,C,fH,fW)."""
    s = p.reshape(f * f, B, H + 1, W + 1, -1)[:, :, :H, :W]
    return F.pixel_shuffle(s.permute(1, 4, 0, 2, 3).reshape(B, -1, H, W), f)


def consumer_image_sums(part, B, H, W, tile_rows=TILE):
    """Per-image channel sums from [tile][segment][quarter][64] partials, reduced the way sres_ca_apply_fwd reads them
    (ca.cu, ca_apply_fwd_kernel): image b takes tiles (b RP) / tile_rows .. ((b+1) RP - 1) / tile_rows, segment 0 of a
    tile that starts inside it, segment 1 of one that starts in the previous image, all four quarters."""
    RP = (H + 1) * (W + 1)
    ts, segs, bs = [], [], []
    for b in range(B):
        for t in range(b * RP // tile_rows, ((b + 1) * RP - 1) // tile_rows + 1):
            ts.append(t)
            segs.append(0 if t * tile_rows >= b * RP else 1)
            bs.append(b)
    idx = [torch.tensor(v, device=part.device) for v in (ts, segs, bs)]
    per = part.double()[idx[0], idx[1]].sum(1)
    return torch.zeros(B, part.shape[-1], dtype=torch.float64, device=part.device).index_add_(0, idx[2], per)


# ---------------------------------------------------------------------------------------------------------------------
# checks
# ---------------------------------------------------------------------------------------------------------------------
def _at(k, shape, dims):
    return "(" + ", ".join(f"{d} {i}" for d, i in zip(dims, np.unravel_index(k, shape))) + ")"


def check(name, got, ref, A, rel_bound, bf16=False, zero=None, dims=("image", "y", "x", "channel")):
    """Element bound 2^-12 A (+ 2^-8 |ref| for a bf16 output), rel-L2 bound, and exact zeros where `zero` is set."""
    g = got.double()
    assert bool(torch.isfinite(g).all()), f"{name}: non-finite value at {_at(int((~torch.isfinite(g)).flatten().nonzero()[0]), g.shape, dims)}"
    d = (g - ref).abs()
    target = ref.float().bfloat16().double() if bf16 else ref
    rel = ((g - target).norm() / ref.norm().clamp_min(1e-300)).item()
    r = d / A.clamp_min(1e-300)
    k = int(r.argmax())
    worst = r.flatten()[k].item()
    print(f"  {name:<46s} rel-L2 {rel:.2e} (bound {rel_bound:.0e})   max|err|/A {worst:.2e} at {_at(k, g.shape, dims)}")
    tol = 2.0 ** -12 * A + (2.0 ** -8 * ref.abs() if bf16 else 0.0)
    bad = (d > tol).flatten()
    if bool(bad.any()):
        k = int(bad.nonzero()[0])
        raise AssertionError(f"{name}: {int(bad.sum())} elements out of bound, first at {_at(k, g.shape, dims)}: got "
                             f"{g.flatten()[k].item():.7e}, ref {ref.flatten()[k].item():.7e}, A {A.flatten()[k].item():.3e}")
    if zero is not None:
        assert bool((g[zero] == 0).all()), f"{name}: masked elements are not exactly 0"
    assert rel < rel_bound, f"{name}: rel-L2 {rel:.3e} >= {rel_bound:.0e}"


def check_ptl(name, p, ref, A, B, H, W, bf16=False, zero=None):
    """A PTL output (without its guard) against NCHW float64 ref / A: padding rows exactly 0, valid rows by `check`."""
    v = p.reshape(B, H + 1, W + 1, -1)
    pads = torch.cat([v[:, H].flatten(), v[:, :H, W].flatten()])
    assert bool((pads == 0).all()), f"{name}: {int((pads != 0).sum())} padding-row elements are not exactly 0"
    check(name, v[:, :H, :W], ref.permute(0, 2, 3, 1), A.permute(0, 2, 3, 1), REL_BF16 if bf16 else REL_F32, bf16,
          None if zero is None else zero.permute(0, 2, 3, 1))


def check_parts(name, part, val, A, B, H, W):
    """POOL / DOT partials: every slot finite; per (image, channel) within 2^-12 of the sum over A of the fp64 sum."""
    assert bool(torch.isfinite(part).all()), f"{name}: non-finite partial-sum slots"
    check(name, consumer_image_sums(part, B, H, W), val.sum((2, 3)), A.sum((2, 3)), REL_SUM, dims=("image", "channel"))


def check_guard(name, buf, n):
    assert bool(torch.isnan(buf[n:].float()).all()), f"{name}: written past its end"


def bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


# ---------------------------------------------------------------------------------------------------------------------
# operands and launches
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    from sres_b200 import _lib as L
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = L.lib()
    lib.sres_conv_pair_flag_bytes.restype = C.c_size_t
    lib.sres_ptl_rows.restype = C.c_int64
    dev = torch.device("cuda:0")
    print(f"\n  device: {torch.cuda.get_device_name(dev)}")
    assert lib.sres_conv_tile_rows(48, 48) == TILE
    return L, lib, dev


@pytest.fixture(autouse=True)
def _release():
    yield
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.synchronize()
        gpu_util._KEEP.clear()


def _gen(dev, *key):
    return torch.Generator(device=dev).manual_seed(zlib.crc32(repr(key).encode()))


def _bf16(g, dev, *shape, scale=1.0):
    return (torch.randn(*shape, device=dev, generator=g) * scale).bfloat16()


def _weights(g, dev, cout, cin=64):
    """bf16-representable fp32 weights of a 3x3 conv, scaled so that outputs stay O(1)."""
    return _bf16(g, dev, cout, cin, 3, 3, scale=(cin * 9) ** -0.5).float()


def _nan(dev, rows, dtype=torch.float32, guard=GUARD):
    return torch.full((rows + guard, 64), NAN, device=dev, dtype=dtype)


def _addend(t):
    """fp32 PTL addend with NaN in its padding rows and a NaN guard: the kernel must zero padding rows, not add them."""
    B, _, H, W = t.shape
    p = to_ptl(t, torch.float32).reshape(B, H + 1, W + 1, 64)
    p[:, H] = NAN
    p[:, :, W] = NAN
    return torch.cat([p.reshape(-1, 64), torch.full((GUARD, 64), NAN, device=t.device)])


def launch(env, a):
    L, lib, _ = env
    L.check(lib.sres_conv3x3_igemm(C.byref(a), L.cur_stream()), "sres_conv3x3_igemm")


def launch_pair(env, a1, a2, flags):
    """conv64_pair of rcan_net.cu: one fused launch when sres_conv_pair_supported takes the pair, else two."""
    L, lib, _ = env
    if lib.sres_conv_pair_supported(C.byref(a1), C.byref(a2)):
        L.check(lib.sres_conv3x3_pair(C.byref(a1), C.byref(a2), ptr(flags), L.cur_stream()), "sres_conv3x3_pair")
        return "fused pair"
    launch(env, a1)
    launch(env, a2)
    return "two launches"


def _flags(env, B, H, W):
    L, lib, dev = env
    return torch.zeros(lib.sres_conv_pair_flag_bytes(B, H, W) // 4, dtype=torch.int32, device=dev)


def _parts(env, B, H, W):
    return torch.full((env[1].sres_conv_mtiles(B, H, W), 2, 4, 64), NAN, device=env[2])


BODY = [pytest.param(64, 48, 48, id="x4-64x48x48"), pytest.param(8, 96, 96, id="x8-8x96x96"),
        pytest.param(5, 10, 11, id="edge-5x10x11"), pytest.param(37, 7, 9, id="edge-37x7x9")]


# ---------------------------------------------------------------------------------------------------------------------
# single identity-mapped 64 -> 64 calls
# ---------------------------------------------------------------------------------------------------------------------
# rcan_net.cu call -> (weights: 0 forward / 1 input gradient, bias, fp32 addend: "own" buffer or "out" = aliased with
# out_f32, second addend (aliased with out_f32), DOT factor + partials (only where (H+1)(W+1) >= 128), outputs)
CALLS = {
    "F2-group-tail": dict(mode=0, bias=True, resid="own", o32=True, o16=True),                # :396
    "F3-body-tail": dict(mode=0, bias=True, resid="own", o16=True),                           # :402 (generic instance)
    "F4-edsr-conv2": dict(mode=0, bias=True, resid="out", o32=True, o16=True),                # :367, r > 0
    "B2-body-tail-dgrad": dict(mode=1, o32=True, o16=True),                                   # :585
    "B3-group-tail-dgrad": dict(mode=1, o32=True, dot=True),                                  # :615
    "B5-first-rcab-dgrad1": dict(mode=1, resid="own", resid2="out", o32=True, o16=True),      # :648
    "B6-edsr-dgrad1": dict(mode=1, resid="out", o32=True, o16=True),                          # :602, r > 0
    "B6-edsr-dgrad1-r0": dict(mode=1, resid="out", o32=True),                                 # :602, r = 0
}


@pytest.mark.gpu
@pytest.mark.parametrize("call", list(CALLS))
@pytest.mark.parametrize("B,H,W", BODY)
def test_conv_call(env, call, B, H, W):
    """One convolution of the RCAB / EDSR / group-tail / body-tail sequence with the epilogue fields rcan_net.cu gives it
    (table CALLS), against fp64.  Measured on a B200: see REL_*."""
    L, lib, dev = env
    c = CALLS[call]
    g = _gen(dev, "call", call, B, H, W)
    rows = B * (H + 1) * (W + 1)
    dot = c.get("dot", False) and (H + 1) * (W + 1) >= TILE
    x = _bf16(g, dev, B, 64, H, W)
    w = _weights(g, dev, 64)
    bias = torch.randn(64, device=dev, generator=g) * 0.5 if c.get("bias") else None
    r1 = torch.randn(B, 64, H, W, device=dev, generator=g) if c.get("resid") else None
    r2 = torch.randn(B, 64, H, W, device=dev, generator=g) if c.get("resid2") else None
    mask = _bf16(g, dev, B, 64, H, W) if dot else None
    xp, wp = to_ptl(x, torch.bfloat16), pack(lib, w, c["mode"])
    maskp = to_ptl(mask, torch.bfloat16) if dot else None
    own = _addend(r1) if c.get("resid") == "own" else None
    out_init = r1 if c.get("resid") == "out" else r2 if c.get("resid2") == "out" else None

    def run():
        o32 = (_addend(out_init) if out_init is not None else _nan(dev, rows)) if c.get("o32") else None
        o16 = _nan(dev, rows, torch.bfloat16) if c.get("o16") else None
        part = _parts(env, B, H, W) if dot else None
        launch(env, conv_args(in_bf16=xp, wpack_bf16=wp, bias=bias, resid_f32=own if own is not None else (o32 if r1 is not None else None),
                              resid2_f32=o32 if r2 is not None else None, mask_bf16=maskp, out_f32=o32, out_bf16=o16,
                              pool_part=part, B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_DOT if dot else 0))
        torch.cuda.synchronize()
        return o32, o16, part

    o32, o16, part = run()
    v, A = conv_ref(x, w if c["mode"] == 0 else dgrad_w(w), bias)
    for r in (r1, r2):
        if r is not None:
            v, A = v + r.double(), A + r.double().abs()
    print(f"\n  {call} {(B, H, W)}")
    if o32 is not None:
        check_ptl("out_f32", o32[:rows], v, A, B, H, W)
        check_guard("out_f32", o32, rows)
    if o16 is not None:
        check_ptl("out_bf16", o16[:rows], v, A, B, H, W, bf16=True)
        check_guard("out_bf16", o16, rows)
    if dot:
        m = mask.double()
        check_parts("dot partials: sum out_f32 * mask", part, v * m, A * m.abs(), B, H, W)
    again = run()
    for a, b in zip((o32, o16, part), again):
        assert a is None or same_bits(a, b), f"{call}: not bit-identical run to run"


# ---------------------------------------------------------------------------------------------------------------------
# the RCAB pairs
# ---------------------------------------------------------------------------------------------------------------------
def fwd_pair_args(env, xp, wp1, b1, wp2, b2, t1, t2, part, B, H, W):
    """rcan_net.cu:383: conv1 bias + ReLU -> bf16 T1; conv2 bias (+ POOL partials when an image covers a tile) -> bf16 T2."""
    L = env[0]
    a1 = conv_args(in_bf16=xp, wpack_bf16=wp1, bias=b1, out_bf16=t1, B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_RELU)
    a2 = conv_args(in_bf16=t1, wpack_bf16=wp2, bias=b2, out_bf16=t2, pool_part=part, B=B, H=H, W=W, n_out=64,
                   epi_flags=L.EPI_POOL if part is not None else 0)
    return a1, a2


def check_fwd_pair(x, w1, b1, w2, b2, t1, t2, part, B, H, W):
    rows = B * (H + 1) * (W + 1)
    pre, A1 = conv_ref(x, w1, b1)
    check_ptl("T1 = relu(conv1 + b1) (bf16)", t1[:rows], pre.clamp_min(0), A1, B, H, W, bf16=True,
              zero=pre < -2.0 ** -12 * A1)
    v2, A2 = conv_ref(ptl_nchw(t1[:rows], B, H, W), w2, b2)
    check_ptl("T2 = conv2 + b2 (bf16)", t2[:rows], v2, A2, B, H, W, bf16=True)
    if part is not None:
        check_parts("pool partials: sum T2", part, v2, A2, B, H, W)
    check_guard("T1", t1, rows)
    check_guard("T2", t2, rows)
    return v2, A2


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", BODY)
def test_rcab_forward_pair(env, B, H, W):
    """F1, the RCAB forward pair (rcan_net.cu:383) through conv64_pair's choice, against fp64: T1 (ReLU-masked elements
    exactly 0), T2 from the kernel's T1, and the POOL partials reduced per image as the channel attention reads them.
    Measured on a B200: see REL_*."""
    L, lib, dev = env
    g = _gen(dev, "fwd pair", B, H, W)
    rows = B * (H + 1) * (W + 1)
    fused = (H + 1) * (W + 1) >= TILE
    x = _bf16(g, dev, B, 64, H, W)
    w1, w2 = _weights(g, dev, 64), _weights(g, dev, 64)
    b1, b2 = torch.randn(64, device=dev, generator=g) * 0.5, torch.randn(64, device=dev, generator=g) * 0.5
    xp, wp1, wp2 = to_ptl(x, torch.bfloat16), pack(lib, w1, 0), pack(lib, w2, 0)
    flags = _flags(env, B, H, W)
    results = []
    for _ in range(2):
        t1, t2 = _nan(dev, rows, torch.bfloat16), _nan(dev, rows, torch.bfloat16)
        part = _parts(env, B, H, W) if fused else None
        how = launch_pair(env, *fwd_pair_args(env, xp, wp1, b1, wp2, b2, t1, t2, part, B, H, W), flags)
        torch.cuda.synchronize()
        assert int(flags.abs().sum()) == 0, "pair flags must be back to all zeros"
        results.append((t1, t2, part))
    print(f"\n  RCAB forward pair {(B, H, W)}: {how}")
    check_fwd_pair(x, w1, b1, w2, b2, *results[0], B, H, W)
    for a, b in zip(*results):
        assert a is None or same_bits(a, b), "not bit-identical run to run"


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", BODY)
def test_rcab_backward_pair(env, B, H, W):
    """B4, the RCAB backward pair (rcan_net.cu:637): dgrad of conv2 masked by T1 > 0 -> bf16 dt1, then dgrad of conv1 added
    into the fp32 gradient trunk in place (out_f32 == resid_f32) with the DOT partials of trunk * T2 of the previous RCAB,
    through conv64_pair's choice (two launches at W = 96), against fp64.  Measured on a B200: see REL_*."""
    L, lib, dev = env
    g = _gen(dev, "bwd pair", B, H, W)
    rows = B * (H + 1) * (W + 1)
    dot = (H + 1) * (W + 1) >= TILE
    dt2 = _bf16(g, dev, B, 64, H, W)
    t1 = _bf16(g, dev, B, 64, H, W).clamp_min(0)
    t2p = _bf16(g, dev, B, 64, H, W)
    trunk = torch.randn(B, 64, H, W, device=dev, generator=g)
    wc2, wc1 = _weights(g, dev, 64), _weights(g, dev, 64)
    dt2p, t1p, t2pp = (to_ptl(t, torch.bfloat16) for t in (dt2, t1, t2p))
    wp2, wp1 = pack(lib, wc2, 1), pack(lib, wc1, 1)
    flags = _flags(env, B, H, W)
    results = []
    for _ in range(2):
        dt1, gb32 = _nan(dev, rows, torch.bfloat16), _addend(trunk)
        part = _parts(env, B, H, W) if dot else None
        a1 = conv_args(in_bf16=dt2p, wpack_bf16=wp2, mask_bf16=t1p, out_bf16=dt1, B=B, H=H, W=W, n_out=64)
        a2 = conv_args(in_bf16=dt1, wpack_bf16=wp1, out_f32=gb32, resid_f32=gb32, mask_bf16=t2pp if dot else None,
                       pool_part=part, B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_DOT if dot else 0)
        how = launch_pair(env, a1, a2, flags)
        torch.cuda.synchronize()
        assert int(flags.abs().sum()) == 0, "pair flags must be back to all zeros"
        results.append((dt1, gb32, part))
    dt1, gb32, part = results[0]
    print(f"\n  RCAB backward pair {(B, H, W)}: {how}")
    keep = (t1 > 0).double()
    v1, A1 = conv_ref(dt2, dgrad_w(wc2))
    check_ptl("dt1 = dgrad2 * (T1 > 0) (bf16)", dt1[:rows], v1 * keep, A1 * keep, B, H, W, bf16=True, zero=keep == 0)
    v2, A2 = conv_ref(ptl_nchw(dt1[:rows], B, H, W), dgrad_w(wc1))
    v2, A2 = v2 + trunk.double(), A2 + trunk.double().abs()
    check_ptl("trunk += dgrad1 (fp32, in place)", gb32[:rows], v2, A2, B, H, W)
    if dot:
        m = t2p.double()
        check_parts("dot partials: sum trunk * T2", part, v2 * m, A2 * m.abs(), B, H, W)
    check_guard("dt1", dt1, rows)
    check_guard("trunk", gb32, rows)
    for a, b in zip(*results):
        assert a is None or same_bits(a, b), "not bit-identical run to run"


@pytest.mark.gpu
def test_rcab_forward_chain_with_channel_attention(env):
    """Four RCABs of a residual group at 64 x 48 x 48 enqueued as rcan_net.cu:383-393 enqueues them, with no host
    synchronisation: pair k (flag buffer k & 1) reads the bf16 trunk the channel attention of RCAB k-1 wrote, and
    sres_ca_apply_fwd reads pair k's POOL partials from the one shared buffer and updates the fp32 trunk in place.
    Every pair's T1 / T2 is bit-identical to the same pair run alone on the same input; T1, T2, save_mean, save_s, the
    bf16 trunk copies and the final trunk match fp64."""
    L, lib, dev = env
    B, H, W, K = 64, 48, 48, 4
    rows = B * (H + 1) * (W + 1)
    g = _gen(dev, "fwd chain")
    x0 = _bf16(g, dev, B, 64, H, W)
    trunk0 = x0.float()        # the head conv writes the fp32 trunk and its bf16 copy; the copy is exact here
    prm = [dict(w1=_weights(g, dev, 64), b1=torch.randn(64, device=dev, generator=g) * 0.5, w2=_weights(g, dev, 64),
                b2=torch.randn(64, device=dev, generator=g) * 0.5,
                cw1=torch.randn(HID, 64, device=dev, generator=g) * 0.3, cb1=torch.randn(HID, device=dev, generator=g),
                cw2=torch.randn(64, HID, device=dev, generator=g) * 0.3, cb2=torch.randn(64, device=dev, generator=g))
           for _ in range(K)]
    for p in prm:
        p["wp1"], p["wp2"] = pack(lib, p["w1"], 0), pack(lib, p["w2"], 0)
    flags = [_flags(env, B, H, W), _flags(env, B, H, W)]
    part = _parts(env, B, H, W)
    xf = to_ptl(trunk0, torch.float32)
    xb = [to_ptl(x0, torch.bfloat16)] + [_nan(dev, rows, torch.bfloat16) for _ in range(K)]
    t1 = [_nan(dev, rows, torch.bfloat16) for _ in range(K)]
    t2 = [_nan(dev, rows, torch.bfloat16) for _ in range(K)]
    mean = torch.full((K, B, 64), NAN, device=dev)
    sv = torch.full((K, B, 64), NAN, device=dev)
    hows = []
    for k, p in enumerate(prm):
        hows.append(launch_pair(env, *fwd_pair_args(env, xb[k], p["wp1"], p["b1"], p["wp2"], p["b2"], t1[k], t2[k], part, B, H, W),
                                flags[k & 1]))
        L.check(lib.sres_ca_apply_fwd(ptr(t2[k]), ptr(part), None, ptr(p["cw1"]), ptr(p["cb1"]), ptr(p["cw2"]), ptr(p["cb2"]),
                                      HID, ptr(xf), ptr(xf), ptr(xb[k + 1]), ptr(mean[k]), ptr(sv[k]), B, H, W,
                                      L.cur_stream()), "sres_ca_apply_fwd")
    torch.cuda.synchronize()
    last_part = part.clone()
    print(f"\n  four RCABs back to back {(B, H, W)}: {', '.join(hows)}")
    assert all(int(f.abs().sum()) == 0 for f in flags), "pair flags must be back to all zeros"
    # fp64: x_{k+1} = x_k + t2_k s_k, every step one fp32 rounding (judged against the sum of |terms| so far)
    xr = to_ptl(trunk0, torch.float32).double()
    S = xr.abs()
    for k, p in enumerate(prm):
        x = ptl_nchw(xb[k][:rows], B, H, W)
        v2, A2 = check_fwd_pair(x, p["w1"], p["b1"], p["w2"], p["b2"], t1[k], t2[k], None, B, H, W)
        m_ref = v2.mean((2, 3))
        check(f"RCAB {k}: save_mean", mean[k], m_ref, A2.mean((2, 3)), REL_SUM, dims=("image", "channel"))
        m = mean[k].double()
        h = torch.relu(m @ p["cw1"].double().T + p["cb1"].double())
        s_ref = torch.sigmoid(h @ p["cw2"].double().T + p["cb2"].double())
        zA = (m.abs() @ p["cw1"].double().abs().T + p["cb1"].double().abs()) @ p["cw2"].double().abs().T + p["cb2"].double().abs()
        check(f"RCAB {k}: save_s (gate of save_mean)", sv[k], s_ref, zA, REL_SUM, dims=("image", "channel"))
        ts = t2[k][:rows].double().reshape(B, -1, 64) * sv[k].double().unsqueeze(1)
        xr = xr + ts.reshape(rows, 64)
        S = S + ts.abs().reshape(rows, 64)
        # A = the fp32 rounding budget of k + 1 steps (2^-24 per step, relative to S); the bf16 rounding is the 2^-8 |ref| term
        check(f"RCAB {k}: bf16 trunk = bf16(x + T2 s)", xb[k + 1][:rows], xr, S * 2.0 ** -12 * (k + 1), REL_BF16, bf16=True,
              dims=("row", "channel"))
        check_guard(f"RCAB {k}: bf16 trunk", xb[k + 1], rows)
    err = (xf.double() - xr).abs()
    print(f"  {'fp32 trunk after four RCABs':<46s} max|err|/sum|terms| {(err / S.clamp_min(1e-300)).max().item():.2e}")
    assert bool((err <= K * 2.0 ** -24 * S).all()), "fp32 trunk is more than one fp32 rounding per step from x + sum T2 s"
    # each pair alone, on the input the chain gave it
    for k, p in enumerate(prm):
        a1, a2 = _nan(dev, rows, torch.bfloat16), _nan(dev, rows, torch.bfloat16)
        pa = _parts(env, B, H, W)
        launch_pair(env, *fwd_pair_args(env, xb[k], p["wp1"], p["b1"], p["wp2"], p["b2"], a1, a2, pa, B, H, W), flags[0])
        torch.cuda.synchronize()
        assert same_bits(a1, t1[k]) and same_bits(a2, t2[k]), f"RCAB {k}: pair differs from the same pair run alone"
        if k == K - 1:
            assert same_bits(pa, last_part), "last pair's partials differ from the same pair run alone"


# ---------------------------------------------------------------------------------------------------------------------
# upsampler and tail
# ---------------------------------------------------------------------------------------------------------------------
UP_FWD = [pytest.param(64, 48, 48, 2, id="x4-stage0-64x48x48"), pytest.param(64, 96, 96, 2, id="x4-stage1-64x96x96"),
          pytest.param(8, 192, 192, 2, id="x8-stage1-8x192x192"), pytest.param(2, 384, 384, 2, id="x8-stage2-2x384x384"),
          pytest.param(16, 48, 48, 3, id="x3-16x48x48"), pytest.param(5, 10, 11, 2, id="edge-5x10x11"),
          pytest.param(37, 7, 9, 3, id="edge-37x7x9-f3")]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W,f", UP_FWD)
def test_upsampler_forward(env, B, H, W, f):
    """F5, an upsampler stage (rcan_net.cu:406): f*f sub-convolutions with PixelShuffle stores (SRES_MAP_SHUFFLE) filling
    one hi-res bf16 PTL, against F.pixel_shuffle of the fp64 64 -> f*f*64 convolution.  384 x 384 leaves one halo-ring
    slot.  Measured on a B200: see REL_*."""
    L, lib, dev = env
    g = _gen(dev, "up fwd", B, H, W, f)
    x = _bf16(g, dev, B, 64, H, W)
    w = _weights(g, dev, f * f * 64)
    b = torch.randn(f * f * 64, device=dev, generator=g) * 0.5
    xp = to_ptl(x, torch.bfloat16)
    subs = [(pack(lib, w, 0, 64, f * f, s), b[s::f * f].contiguous()) for s in range(f * f)]
    rows_hi = lib.sres_ptl_rows(B, f * H, f * W)

    def run():
        out = _nan(dev, rows_hi, torch.bfloat16)
        for s, (wp, bs) in enumerate(subs):
            launch(env, conv_args(in_bf16=xp, wpack_bf16=wp, bias=bs, out_bf16=out, B=B, H=H, W=W, n_out=64,
                                  map_mode=L.MAP_SHUFFLE, sub_i=s // f, sub_j=s % f, shuffle_factor=f))
        torch.cuda.synchronize()
        return out

    out = run()
    v, A = conv_ref(x, w, b)
    print(f"\n  upsampler forward {(B, H, W)} x{f}")
    check_ptl("hi-res PTL (bf16)", out[:rows_hi], F.pixel_shuffle(v, f), F.pixel_shuffle(A, f), B, f * H, f * W, bf16=True)
    check_guard("hi-res PTL", out, rows_hi)
    assert same_bits(out, run()), "not bit-identical run to run"


TAIL = [pytest.param(64, 192, 192, 2, id="x4-64x192x192"), pytest.param(2, 768, 768, 4, id="x8-2x768x768"),
        pytest.param(5, 10, 11, 16, id="edge-5x10x11"), pytest.param(37, 7, 9, 3, id="edge-37x7x9")]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W,cout", TAIL)
def test_tail_conv(env, B, H, W, cout):
    """F6, the tail convolution (rcan_net.cu:412): 16 packed output rows, bias gathered to 16, c_real real channels into
    planar fp32 (out_nchw), against fp64.  Measured on a B200: see REL_*."""
    L, lib, dev = env
    g = _gen(dev, "tail", B, H, W, cout)
    x = _bf16(g, dev, B, 64, H, W)
    w = _weights(g, dev, cout)
    b = torch.randn(cout, device=dev, generator=g) * 0.5
    b16 = torch.cat([b, torch.zeros(16 - cout, device=dev)])
    xp, wp = to_ptl(x, torch.bfloat16), pack(lib, w, 0, 16)
    assert lib.sres_conv_supported(H, W, 16)
    n = B * cout * H * W

    def run():
        out = torch.full((n + GUARD * 64,), NAN, device=dev)
        launch(env, conv_args(in_bf16=xp, wpack_bf16=wp, bias=b16, out_nchw=out, c_real=cout, B=B, H=H, W=W, n_out=16))
        torch.cuda.synchronize()
        return out

    out = run()
    v, A = conv_ref(x, w, b)
    print(f"\n  tail conv {(B, H, W)} -> {cout} channels")
    check("out_nchw", out[:n].reshape(B, cout, H, W), v, A, REL_F32, dims=("image", "channel", "y", "x"))
    check_guard("out_nchw", out, n)
    assert same_bits(out, run()), "not bit-identical run to run"


def up_dgrad_stage(env, dy, wps, B, H, W, f, sf, acc32, acc16):
    """rcan_net.cu:574-580: the f*f input-gradient sub-convolutions of one upsampler stage, sub-grid `sub` of dy (the
    output gradient in PixelUnshuffle layout) through the packed dgrad weights of sub-convolution `sub`; out_f32 = acc32
    (its addend from the second sub on), bf16 acc16 on the last; UNSHUFFLE(sf) store for stage > 0 (sf given)."""
    L = env[0]
    rows = B * (H + 1) * (W + 1)
    for s, wp in enumerate(wps):
        launch(env, conv_args(in_bf16=dy[s * rows:(s + 1) * rows], wpack_bf16=wp, out_f32=acc32, resid_f32=acc32 if s else None,
                              out_bf16=acc16 if s == f * f - 1 else None, B=B, H=H, W=W, n_out=64,
                              map_mode=L.MAP_UNSHUFFLE if sf else L.MAP_IDENT, shuffle_factor=sf or 2))


def check_unshuffle_pads(name, p, B, H, W, sf):
    """Sub-grid (si, sj) of an UNSHUFFLE store gets its padding row written (0) only when si == 0 and its padding column
    only when sj == 0; the others keep whatever the buffer held (0 or the NaN sentinel)."""
    v = p.reshape(sf * sf, B, H + 1, W + 1, -1).float()
    for s in range(sf * sf):
        si, sj = divmod(s, sf)
        for piece, written in ((v[s, :, H, :W], si == 0), (v[s, :, :H, W], sj == 0), (v[s, :, H, W], si == 0 and sj == 0)):
            ok = (piece == 0) if written else ((piece == 0) | torch.isnan(piece))
            assert bool(ok.all()), f"{name}: padding of sub-grid {s} holds something other than {'0' if written else '0 / NaN'}"


def check_up_dgrad(name, acc32, acc16, dU, w, B, H, W, f, sf):
    """Stage output against fp64: dx = conv of pixel_unshuffle(dU, f) with the dgrad weights of the 64 -> f*f*64 conv."""
    v, A = conv_ref(F.pixel_unshuffle(dU.double(), f), dgrad_w(w))
    if sf is None:
        rows = B * (H + 1) * (W + 1)
        check_ptl(f"{name} out_f32", acc32[:rows], v, A, B, H, W)
        check_ptl(f"{name} out_bf16", acc16[:rows], v, A, B, H, W, bf16=True)
    else:
        Hl, Wl = H // sf, W // sf
        rows = sf * sf * B * (Hl + 1) * (Wl + 1)
        for t, bf in ((acc32, False), (acc16, True)):
            tag = f"{name} {'out_bf16' if bf else 'out_f32'} (unshuffled)"
            check_unshuffle_pads(tag, t[:rows], B, Hl, Wl, sf)
            got = from_unshuffle_ptl(t[:rows], B, Hl, Wl, sf)
            check(tag, got.permute(0, 2, 3, 1), v.permute(0, 2, 3, 1), A.permute(0, 2, 3, 1), REL_BF16 if bf else REL_F32, bf)
    check_guard(f"{name} out_f32", acc32, rows)
    check_guard(f"{name} out_bf16", acc16, rows)


UP_DGRAD = [pytest.param(2, 384, 384, 2, 2, id="x8-stage2-2x384x384-unshuffle"),
            pytest.param(8, 96, 96, 2, None, id="x8-stage0-8x96x96"),
            pytest.param(16, 48, 48, 3, None, id="x3-16x48x48"),
            pytest.param(5, 20, 22, 2, 2, id="edge-5x20x22-unshuffle"),
            pytest.param(5, 10, 11, 2, None, id="edge-5x10x11"),
            pytest.param(37, 7, 9, 3, None, id="edge-37x7x9-f3")]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W,f,sf", UP_DGRAD)
def test_upsampler_dgrad(env, B, H, W, f, sf):
    """B1, one upsampler stage of the backward (rcan_net.cu:574) against fp64: stage > 0 stores UNSHUFFLE(sf) into the
    previous level's sub-grids (the sub-grid padding the store leaves unwritten may hold 0 or the NaN sentinel), stage 0
    stores in place.  Measured on a B200: see REL_*."""
    L, lib, dev = env
    g = _gen(dev, "up dgrad", B, H, W, f, sf)
    dU = _bf16(g, dev, B, 64, f * H, f * W)
    w = _weights(g, dev, f * f * 64)
    dy = unshuffle_ptl(dU, f, torch.bfloat16)
    wps = [pack(lib, w, 1, 64, f * f, s) for s in range(f * f)]
    out_rows = B * (H + 1) * (W + 1) if sf is None else sf * sf * B * (H // sf + 1) * (W // sf + 1)

    def run():
        acc32, acc16 = _nan(dev, out_rows), _nan(dev, out_rows, torch.bfloat16)
        up_dgrad_stage(env, dy, wps, B, H, W, f, sf, acc32, acc16)
        torch.cuda.synchronize()
        return acc32, acc16

    acc32, acc16 = run()
    print(f"\n  upsampler dgrad {(B, H, W)} x{f}, {'UNSHUFFLE(%d)' % sf if sf else 'IDENT'}")
    check_up_dgrad("stage", acc32, acc16, dU, w, B, H, W, f, sf)
    for a, b in zip((acc32, acc16), run()):
        assert same_bits(a, b), "not bit-identical run to run"


@pytest.mark.gpu
def test_upsampler_dgrad_chain_x4(env):
    """B1 of the x4 backward at B = 64 as rcan_net.cu:565-581 enqueues it, with no host synchronisation: stage 1 (four
    sub-convolutions at 96 x 96, UNSHUFFLE(2) into 48 x 48 sub-grids), then stage 0 (four sub-convolutions at 48 x 48,
    IDENT) reading stage 1's bf16 result.  The sub-grid buffers start zero-filled in their padding rows and NaN elsewhere,
    as the once-zeroed workspace leaves them.  Each stage against fp64 from the operands it read."""
    L, lib, dev = env
    B, H = 64, 48
    g = _gen(dev, "up dgrad chain")
    dU2 = _bf16(g, dev, B, 64, 4 * H, 4 * H)
    w1, w0 = _weights(g, dev, 256), _weights(g, dev, 256)
    dy1 = unshuffle_ptl(dU2, 2, torch.bfloat16)
    wps1 = [pack(lib, w1, 1, 64, 4, s) for s in range(4)]
    wps0 = [pack(lib, w0, 1, 64, 4, s) for s in range(4)]
    rows0 = B * (H + 1) * (H + 1)
    du32 = to_ptl(torch.full((4 * B, 64, H, H), NAN, device=dev), torch.float32)
    du16 = to_ptl(torch.full((4 * B, 64, H, H), NAN, device=dev), torch.bfloat16)
    du32 = torch.cat([du32, torch.full((GUARD, 64), NAN, device=dev)])
    du16 = torch.cat([du16, torch.full((GUARD, 64), NAN, device=dev, dtype=torch.bfloat16)])
    dres32, dres16 = _nan(dev, rows0), _nan(dev, rows0, torch.bfloat16)
    up_dgrad_stage(env, dy1, wps1, B, 2 * H, 2 * H, 2, 2, du32, du16)
    up_dgrad_stage(env, du16, wps0, B, H, H, 2, None, dres32, dres16)
    torch.cuda.synchronize()
    print(f"\n  x4 upsampler backward chain, B = {B}")
    check_up_dgrad("stage 1 (96 -> UNSHUFFLE 48)", du32, du16, dU2, w1, B, 2 * H, 2 * H, 2, 2)
    dU1 = from_unshuffle_ptl(du16[:4 * rows0], B, H, H, 2)      # what stage 0 read
    check_up_dgrad("stage 0 (48, IDENT)", dres32, dres16, dU1, w0, B, H, H, 2, None)


# ---------------------------------------------------------------------------------------------------------------------
# the references themselves (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_reference_helpers_cpu():
    """The fp64 references and layout builders above against F.conv2d / F.conv_transpose2d / pixel (un)shuffle and the
    layouts include/sres_b200.h defines, in float64 on the CPU at tiny sizes: a wrong reference fails here, not on the GPU."""
    g = torch.Generator().manual_seed(7)
    B, H, W, f = 3, 5, 4, 2
    x = torch.randn(B, 64, H, W, generator=g, dtype=torch.float64)
    w = torch.randn(8, 64, 3, 3, generator=g, dtype=torch.float64)
    b = torch.randn(8, generator=g, dtype=torch.float64)
    y, A = conv_ref(x, w, b)
    assert torch.allclose(y, F.conv2d(x, w, b, padding=1), rtol=1e-12, atol=1e-12)
    assert torch.allclose(A, F.conv2d(x.abs(), w.abs(), b.abs(), padding=1), rtol=1e-12, atol=1e-12)
    dy = torch.randn(B, 8, H, W, generator=g, dtype=torch.float64)
    dx, _ = conv_ref(dy, dgrad_w(w))
    assert torch.allclose(dx, F.conv_transpose2d(dy, w, padding=1), rtol=1e-12, atol=1e-12)
    # dgrad of the 64 -> f*f*64 upsampler conv through pixel_unshuffle = the autograd input gradient of conv + pixel_shuffle
    wu = torch.randn(f * f * 64, 64, 3, 3, generator=g, dtype=torch.float64)
    xr = x.clone().requires_grad_(True)
    dU = torch.randn(B, 64, f * H, f * W, generator=g, dtype=torch.float64)
    (F.pixel_shuffle(F.conv2d(xr, wu, padding=1), f) * dU).sum().backward()
    dxu, _ = conv_ref(F.pixel_unshuffle(dU, f), dgrad_w(wu))
    assert torch.allclose(dxu, xr.grad, rtol=1e-10, atol=1e-10)
    # sub-convolution s = i*f + j of the upsampler (packed with oc_stride f*f, oc_offset s) lands at (f y + i, f x + j)
    full, _ = conv_ref(x, wu)
    up = F.pixel_shuffle(full, f)
    for s in range(f * f):
        sub, _ = conv_ref(x, wu[s::f * f])
        assert torch.equal(up[:, :, s // f::f, s % f::f], sub)
    # PTL: position (b, y, x) at row b (H+1)(W+1) + y (W+1) + x, padding rows 0
    p = to_ptl(x, torch.float64)
    for bb, yy, xx in ((0, 0, 0), (2, 4, 3), (1, 2, 1)):
        assert torch.equal(p[bb * (H + 1) * (W + 1) + yy * (W + 1) + xx], x[bb, :, yy, xx])
    v = p.reshape(B, H + 1, W + 1, 64)
    assert bool((v[:, H] == 0).all() and (v[:, :, W] == 0).all())
    assert torch.equal(ptl_nchw(p, B, H, W), x)
    # PixelUnshuffle layout: hi-res (b, y, x) -> sub-grid (y % f) f + (x % f), position (b, y / f, x / f)
    hi = torch.randn(B, 64, f * H, f * W, generator=g, dtype=torch.float64)
    u = unshuffle_ptl(hi, f, torch.float64)
    rows = B * (H + 1) * (W + 1)
    assert u.shape[0] == f * f * rows
    for bb in range(B):
        for yy in range(f * H):
            for xx in range(f * W):
                s = (yy % f) * f + xx % f
                assert torch.equal(u[s * rows + bb * (H + 1) * (W + 1) + (yy // f) * (W + 1) + xx // f], hi[bb, :, yy, xx])
    assert torch.equal(from_unshuffle_ptl(u, B, H, W, f), hi)
    # the consumer's per-image reduction of [tile][segment][quarter][64] partials, from per-row values spread over tiles,
    # segments and quarters as the conv epilogue spreads them (tiles that straddle two images: 5 x 10 x 11)
    for B2, H2, W2 in ((5, 10, 11), (4, 12, 12), (2, 20, 24)):
        RP = (H2 + 1) * (W2 + 1)
        n = B2 * RP
        val = torch.randn(n, 64, generator=g, dtype=torch.float64)
        q = torch.arange(n)
        t = q // TILE
        seg = q // RP - (t * TILE) // RP
        assert int(seg.max()) <= 1
        nt = (n + TILE - 1) // TILE
        part = torch.zeros(nt * 8, 64, dtype=torch.float64).index_add_(0, (t * 2 + seg) * 4 + (q % 128) // 32, val)
        got = consumer_image_sums(part.reshape(nt, 2, 4, 64), B2, H2, W2)
        assert torch.allclose(got, val.reshape(B2, RP, 64).sum(1), rtol=1e-12, atol=1e-12)
