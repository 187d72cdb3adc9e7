"""GPU parity tests, kernel by kernel, through the C ABI, against the CPU oracle's arithmetic
(plain fp32 PyTorch ops on the CPU -- the reference's own math).  Tolerances: the tensor-core kernels
take bf16 operands with fp32 accumulation, so they are compared with fp32 math on the SAME
bf16-rounded operands at 2e-3 relative (accumulation order only); fp32 kernels at 1e-5."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rcan_oracle as O
from gpu_util import (bf16_round, check_grad, conv3x3_wgrad_ref, conv_args, from_ptl, pack, pads_are_zero, ptr, rel_l2, run_conv,
                      to_ptl)

pytestmark = pytest.mark.gpu
GEOMS = [(1, 48, 48), (3, 20, 24), (2, 5, 7), (2, 96, 96), (5, 12, 12)]


@pytest.fixture(scope="module")
def env():
    from sres_b200 import _lib as L
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.manual_seed(1234)
    return L, L.lib(), torch.device("cuda:0")


def _rand(dev, *shape, scale=1.0):
    return bf16_round(torch.randn(*shape) * scale), None


@pytest.mark.parametrize("B,H,W", GEOMS)
def test_conv_forward_bias_relu_pool(env, B, H, W):
    L, lib, dev = env
    x = bf16_round(torch.randn(B, 64, H, W))
    w = bf16_round(torch.randn(64, 64, 3, 3) * 0.05)
    b = torch.randn(64)
    ref = F.relu(F.conv2d(x, w, b, padding=1))
    xp = to_ptl(x.to(dev), torch.bfloat16)
    rows = xp.shape[0]
    out32 = torch.full((rows, 64), float("nan"), device=dev)
    out16 = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
    nt = lib.sres_conv_mtiles(B, H, W)
    pool = torch.full((nt, 2, 4, 64), float("nan"), device=dev)
    fused = (H + 1) * (W + 1) >= 128
    wp, bd = pack(lib, w.to(dev), 0), b.to(dev)
    a = conv_args(in_bf16=xp, wpack_bf16=wp, bias=bd, out_bf16=out16, B=B, H=H, W=W, n_out=64,
                  epi_flags=L.EPI_RELU | (L.EPI_POOL if fused else 0))
    if fused:
        a.pool_part = pool.data_ptr()
    run_conv(lib, a)
    run_conv(lib, conv_args(in_bf16=xp, wpack_bf16=wp, bias=bd, out_f32=out32, B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_RELU))
    assert pads_are_zero(out32, B, H, W) and pads_are_zero(out16, B, H, W)
    assert rel_l2(from_ptl(out32, B, H, W).cpu(), ref) < 2e-3
    assert rel_l2(from_ptl(out16, B, H, W).cpu(), ref) < 6e-3          # + one bf16 rounding of the output
    if fused:
        assert torch.isfinite(pool).all()
        assert rel_l2(image_sums(pool, B, H, W, lib.sres_conv_tile_rows(H, W)), ref.sum((2, 3))) < 1e-4


def image_sums(part, B, H, W, tile_rows):
    """[tile][segment][lane quarter][64] per-tile partial sums -> per-image channel sums [B][64]."""
    RP = (H + 1) * (W + 1)
    pc = part.detach().cpu().nan_to_num(0.0)
    sums = torch.zeros(B, 64)
    for t in range(pc.shape[0]):
        b0 = (t * tile_rows) // RP
        for seg in range(2):
            if b0 + seg < B and t * tile_rows < B * RP:
                sums[b0 + seg] += pc[t, seg].sum(0)
    return sums


@pytest.mark.parametrize("B,H,W", [(3, 20, 24), (5, 48, 48), (64, 48, 48), (2, 96, 96)])
def test_conv_pair_equals_two_launches(env, B, H, W):
    """The fused two-convolution launch (phase 2 reads phase 1's tiles behind per-tile ready counters) computes exactly what
    the two separate launches compute -- same MMAs, same epilogue arithmetic: every output bit-equal, per-tile partial
    sums bit-equal -- for the RCAB forward pair (conv1 -> conv2 + pool) and the backward pair (dgrad2 -> dgrad1 with the
    fp32 read-modify-write and the sum g*t2).  Repeated launches on one flag buffer check that the counters clean
    themselves (all zero afterwards) and that nothing depends on timing."""
    L, lib, dev = env
    lib.sres_conv_pair_flag_bytes.restype = C.c_size_t
    rows = lib.sres_ptl_rows(B, H, W)
    nt = (rows + 127) // 128
    flags = torch.zeros(lib.sres_conv_pair_flag_bytes(B, H, W) // 4, dtype=torch.int32, device=dev)
    xin = to_ptl(bf16_round(torch.randn(B, 64, H, W)).to(dev), torch.bfloat16)
    t1m = to_ptl(torch.randn(B, 64, H, W).to(dev), torch.bfloat16)
    t2f = to_ptl(torch.randn(B, 64, H, W).to(dev), torch.bfloat16)
    trunk = to_ptl(torch.randn(B, 64, H, W).to(dev), torch.float32)
    w1 = pack(lib, (torch.randn(64, 64, 3, 3) * 0.05).to(dev), 0)
    w2 = pack(lib, (torch.randn(64, 64, 3, 3) * 0.05).to(dev), 1)
    b1, b2 = torch.randn(64, device=dev), torch.randn(64, device=dev)

    def bufs():
        return dict(mid=torch.full((rows, 64), float("nan"), device=dev, dtype=torch.bfloat16),
                    o16=torch.full((rows, 64), float("nan"), device=dev, dtype=torch.bfloat16),
                    o32=trunk.clone(), part=torch.full((nt, 2, 4, 64), float("nan"), device=dev))

    def fwd_args(bf):
        a1 = conv_args(in_bf16=xin, wpack_bf16=w1, bias=b1, out_bf16=bf["mid"], B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_RELU)
        a2 = conv_args(in_bf16=bf["mid"], wpack_bf16=w2, bias=b2, out_bf16=bf["o16"], pool_part=bf["part"], B=B, H=H, W=W, n_out=64,
                       epi_flags=L.EPI_POOL)
        return a1, a2

    def bwd_args(bf):
        a1 = conv_args(in_bf16=xin, wpack_bf16=w1, mask_bf16=t1m, out_bf16=bf["mid"], B=B, H=H, W=W, n_out=64)
        a2 = conv_args(in_bf16=bf["mid"], wpack_bf16=w2, mask_bf16=t2f, out_f32=bf["o32"], resid_f32=bf["o32"], pool_part=bf["part"],
                       B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_DOT)
        return a1, a2

    for name, mk in (("forward pair", fwd_args), ("backward pair", bwd_args)):
        ref = bufs()
        a1, a2 = mk(ref)
        run_conv(lib, a1)
        run_conv(lib, a2)
        for rep in range(6):
            got = bufs()
            a1, a2 = mk(got)
            if not lib.sres_conv_pair_supported(C.byref(a1), C.byref(a2)):
                assert W > 62 and name == "backward pair"     # wide halo ring + 64 KB of epilogue slabs do not fit: two launches
                break
            L.check(lib.sres_conv3x3_pair(C.byref(a1), C.byref(a2), ptr(flags), L.cur_stream()), "sres_conv3x3_pair")
            torch.cuda.synchronize()
            assert int(flags.abs().sum()) == 0, (name, rep, "ready / consumed counters must reset themselves")
            for k in ("mid", "o16", "o32", "part"):
                a, b = got[k], ref[k]
                assert torch.equal(a.float().nan_to_num(7.0), b.float().nan_to_num(7.0)), (name, rep, k)


@pytest.mark.parametrize("B,H,W", [(3, 20, 24), (5, 48, 48)])
def test_conv_epilogue_flavours_agree(env, B, H, W):
    """The tap-per-MMA kernel's compile-time epilogue flavours (fragment-layout column sums for the pooled / dot-product
    ones) and the generic runtime-flag kernel (debug flag 16, row-layout column sums) compute the same thing: outputs
    bit-equal, per-tile partial sums equal up to summation order."""
    L, lib, dev = env
    rows = lib.sres_ptl_rows(B, H, W)
    nt = lib.sres_conv_mtiles(B, H, W)
    xin = to_ptl(bf16_round(torch.randn(B, 64, H, W)).to(dev), torch.bfloat16)
    msk = to_ptl(torch.randn(B, 64, H, W).to(dev), torch.bfloat16)
    trunk = to_ptl(torch.randn(B, 64, H, W).to(dev), torch.float32)
    wp = pack(lib, (torch.randn(64, 64, 3, 3) * 0.05).to(dev), 0)
    bias = torch.randn(64, device=dev)
    flavours = {
        "conv1": dict(bias=bias, epi_flags=L.EPI_RELU, o16=True),
        "conv2": dict(bias=bias, epi_flags=L.EPI_POOL, o16=True, part=True),
        "dgrad2": dict(mask_bf16=msk, o16=True),
        "dgrad1": dict(mask_bf16=msk, epi_flags=L.EPI_DOT, o32=True, rmw=True, part=True),
        "group dgrad": dict(mask_bf16=msk, epi_flags=L.EPI_DOT, o32=True, part=True),
    }
    for name, f in flavours.items():
        results = []
        for dbg in (0, 16):
            out16 = torch.full((rows, 64), float("nan"), device=dev, dtype=torch.bfloat16)
            out32 = trunk.clone() if f.get("rmw") else torch.full((rows, 64), float("nan"), device=dev)
            part = torch.full((nt, 2, 4, 64), float("nan"), device=dev)
            kw = dict(in_bf16=xin, wpack_bf16=wp, B=B, H=H, W=W, n_out=64, epi_flags=f.get("epi_flags", 0), debug_flags=dbg)
            for k in ("bias", "mask_bf16"):
                if k in f:
                    kw[k] = f[k]
            if f.get("o16"):
                kw["out_bf16"] = out16
            if f.get("o32"):
                kw["out_f32"] = out32
            if f.get("rmw"):
                kw["resid_f32"] = out32
            if f.get("part"):
                kw["pool_part"] = part
            run_conv(lib, conv_args(**kw))
            results.append((out16 if f.get("o16") else out32, part))
        ref_out, ref_part = results[0]
        assert torch.isfinite(ref_out.float()).all(), name
        for out, part in results[1:]:
            assert torch.equal(out, ref_out), name
            if f.get("part"):
                # [tile][segment][lane quarter][64]: the second segment only exists for tiles that straddle two images
                assert rel_l2(part.nan_to_num(0.0).sum(2), ref_part.nan_to_num(0.0).sum(2)) < 1e-5, name


@pytest.mark.parametrize("B,H,W", GEOMS[:3])
def test_conv_dgrad_mask_residuals(env, B, H, W):
    """Input gradient = conv with transposed/flipped weights; ReLU-backward mask; two fp32 addends."""
    L, lib, dev = env
    dy = bf16_round(torch.randn(B, 64, H, W))
    w = bf16_round(torch.randn(64, 64, 3, 3) * 0.05)
    t1 = bf16_round(torch.randn(B, 64, H, W)).clamp_min(0)
    r1, r2 = torch.randn(B, 64, H, W), torch.randn(B, 64, H, W)
    dx = F.conv_transpose2d(dy, w, None, padding=1)
    ref_mask = dx * (t1 > 0)
    ref_res = dx + r1 + r2
    dyp = to_ptl(dy.to(dev), torch.bfloat16)
    wp = pack(lib, w.to(dev), 1)
    out16 = torch.zeros(dyp.shape[0], 64, device=dev, dtype=torch.bfloat16)
    run_conv(lib, conv_args(in_bf16=dyp, wpack_bf16=wp, mask_bf16=to_ptl(t1.to(dev), torch.bfloat16), out_bf16=out16,
                            B=B, H=H, W=W, n_out=64))
    assert rel_l2(from_ptl(out16, B, H, W).cpu(), ref_mask) < 6e-3 and pads_are_zero(out16, B, H, W)
    acc = to_ptl(r1.to(dev), torch.float32)
    run_conv(lib, conv_args(in_bf16=dyp, wpack_bf16=wp, resid_f32=acc, resid2_f32=to_ptl(r2.to(dev), torch.float32), out_f32=acc,
                            B=B, H=H, W=W, n_out=64))
    assert rel_l2(from_ptl(acc, B, H, W).cpu(), ref_res) < 2e-3 and pads_are_zero(acc, B, H, W)
    if (H + 1) * (W + 1) >= 128:
        # fused channel-attention backward reduction: per-tile sums of out * other (SRES_EPI_DOT)
        nt = lib.sres_conv_mtiles(B, H, W)
        part = torch.full((nt, 2, 4, 64), float("nan"), device=dev)
        out32 = torch.zeros(dyp.shape[0], 64, device=dev)
        run_conv(lib, conv_args(in_bf16=dyp, wpack_bf16=wp, mask_bf16=to_ptl(t1.to(dev), torch.bfloat16), out_f32=out32,
                                pool_part=part, B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_DOT))
        assert rel_l2(from_ptl(out32, B, H, W).cpu(), dx) < 2e-3          # the mask operand must NOT gate the output
        assert torch.isfinite(part).all()
        assert rel_l2(image_sums(part, B, H, W, lib.sres_conv_tile_rows(H, W)), (dx * t1).sum((2, 3))) < 2e-3


@pytest.mark.parametrize("f", [2, 3])
def test_upsampler_conv_pixelshuffle_and_back(env, f):
    """conv 64->f*f*64 + PixelShuffle(f) as f*f sub-convs with shuffled stores (blocks.py:62-73), and the
    inverse addressing used by the backward pass."""
    L, lib, dev = env
    B, H, W = 2, 12, 10
    x = bf16_round(torch.randn(B, 64, H, W))
    w = bf16_round(torch.randn(f * f * 64, 64, 3, 3) * 0.05)
    b = torch.randn(f * f * 64)
    ref = F.pixel_shuffle(F.conv2d(x, w, b, padding=1), f)
    xp = to_ptl(x.to(dev), torch.bfloat16)
    lib.sres_ptl_rows.restype = C.c_int64
    out16 = torch.full((lib.sres_ptl_rows(B, f * H, f * W), 64), float("nan"), device=dev, dtype=torch.bfloat16)
    for sub in range(f * f):
        bsub = b[sub::f * f].contiguous().to(dev)
        run_conv(lib, conv_args(in_bf16=xp, wpack_bf16=pack(lib, w.to(dev), 0, 64, f * f, sub), bias=bsub, out_bf16=out16,
                                B=B, H=H, W=W, n_out=64, map_mode=L.MAP_SHUFFLE, sub_i=sub // f, sub_j=sub % f, shuffle_factor=f))
    assert torch.isfinite(out16.float()).all() and pads_are_zero(out16, B, f * H, f * W)
    assert rel_l2(from_ptl(out16, B, f * H, f * W).cpu(), ref) < 6e-3
    # unshuffle store: identity-weight conv of the hi-res tensor lands in f*f low-res sub-grids
    hi = bf16_round(torch.randn(B, 64, f * H, f * W))
    wid = torch.zeros(64, 64, 3, 3)
    wid[torch.arange(64), torch.arange(64), 1, 1] = 1.0
    rows_lo = lib.sres_ptl_rows(B, H, W)
    sub16 = torch.zeros(f * f * rows_lo, 64, device=dev, dtype=torch.bfloat16)
    run_conv(lib, conv_args(in_bf16=to_ptl(hi.to(dev), torch.bfloat16), wpack_bf16=pack(lib, wid.to(dev), 0), out_bf16=sub16,
                            B=B, H=f * H, W=f * W, n_out=64, map_mode=L.MAP_UNSHUFFLE, shuffle_factor=f))
    un = F.pixel_unshuffle(hi, f).reshape(B, 64, f * f, H, W)
    for sub in range(f * f):
        got = from_ptl(sub16[sub * rows_lo:(sub + 1) * rows_lo], B, H, W).cpu()
        assert torch.equal(got, un[:, :, sub])


@pytest.mark.parametrize("n128", ["0"])
@pytest.mark.parametrize("B,H,W", GEOMS[:4])
def test_conv_wgrad(env, B, H, W, n128):
    """One-job weight gradient against fp64 on the same bf16 operands: products are exact in fp32, only the summation order
    differs.  Bounds at ~10x the rel-L2 measured on a B200 (dw <= 2.5e-7, db <= 1.7e-7), every element within 2^-12 of its |x||dy| sum."""
    L, lib, dev = env
    lib.sres_conv_wgrad_workspace_bytes.restype = C.c_size_t
    x = bf16_round(torch.randn(B, 64, H, W))
    dy = bf16_round(torch.randn(B, 64, H, W))
    ref, A = conv3x3_wgrad_ref(x, dy)
    refb, Ab = dy.double().sum((0, 2, 3)), dy.double().abs().sum((0, 2, 3))
    wsb = lib.sres_conv_wgrad_workspace_bytes()
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    dw = torch.full((64, 64, 3, 3), float("nan"), device=dev)
    db = torch.full((64,), float("nan"), device=dev)
    xp, dyp = to_ptl(x.to(dev), torch.bfloat16), to_ptl(dy.to(dev), torch.bfloat16)

    def run(acc):
        L.check(lib.sres_conv3x3_wgrad(ptr(xp), ptr(dyp), B, H, W, ptr(dw), ptr(db), 64, 1, 0, acc, ptr(ws),
                                       C.c_size_t(wsb), L.cur_stream()), "wgrad")
        torch.cuda.synchronize()
    run(0)
    check_grad("dw", dw.cpu(), ref, A, 3e-6)
    check_grad("db", db.cpu(), refb, Ab, 2e-6)
    first = dw.clone()
    run(0)
    assert torch.equal(dw, first), "wgrad must be deterministic run to run"
    run(1)
    check_grad("dw, accumulate = 1", dw.cpu(), 2 * ref, 2 * A, 3e-6)


def test_head_and_tail_convs(env):
    """Cin->64 head conv, 64->Cout tail conv (tensor cores, N padded to 16), their gradients."""
    L, lib, dev = env
    lib.sres_small_wgrad_workspace_bytes.restype = C.c_size_t
    wsb = lib.sres_small_wgrad_workspace_bytes()
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    for Cs, B, H, W in [(2, 3, 20, 24), (1, 2, 9, 9), (4, 1, 16, 12)]:
        x = torch.randn(B, Cs, H, W)
        w, b = torch.randn(64, Cs, 3, 3) * 0.2, torch.randn(64)
        ref = F.conv2d(x, w, b, padding=1)
        rows = B * (H + 1) * (W + 1)
        o32 = torch.full((rows, 64), float("nan"), device=dev)
        o16 = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
        xd = x.to(dev)
        L.check(lib.sres_conv3x3_small_in(ptr(xd), ptr(w.to(dev)), ptr(b.to(dev)), B, Cs, H, W, 0, 0, ptr(o32), ptr(o16),
                                          L.cur_stream()), "head")
        torch.cuda.synchronize()
        assert rel_l2(from_ptl(o32, B, H, W).cpu(), ref) < 1e-5 and pads_are_zero(o32, B, H, W) and pads_are_zero(o16, B, H, W)
        # head wgrad with two gradient addends
        g1, g2 = torch.randn(B, 64, H, W), torch.randn(B, 64, H, W)
        dw = torch.empty(64, Cs, 3, 3, device=dev)
        db = torch.empty(64, device=dev)
        L.check(lib.sres_small_in_wgrad(ptr(to_ptl(g1.to(dev), torch.float32)), ptr(to_ptl(g2.to(dev), torch.float32)), ptr(xd),
                                        B, Cs, H, W, ptr(dw), ptr(db), 0, ptr(ws), C.c_size_t(wsb), L.cur_stream()), "head wgrad")
        torch.cuda.synchronize()
        assert rel_l2(dw.cpu(), torch.nn.grad.conv2d_weight(x, (64, Cs, 3, 3), g1 + g2, padding=1)) < 1e-4
        assert rel_l2(db.cpu(), (g1 + g2).sum((0, 2, 3))) < 1e-4
        # tail conv forward 64 -> Cs on the tensor cores
        u = bf16_round(torch.randn(B, 64, H, W))
        wt, bt = bf16_round(torch.randn(Cs, 64, 3, 3) * 0.05), torch.randn(Cs)
        up = to_ptl(u.to(dev), torch.bfloat16)
        bias16 = torch.zeros(16, device=dev)
        bias16[:Cs] = bt.to(dev)
        out = torch.full((B, Cs, H, W), float("nan"), device=dev)
        run_conv(lib, conv_args(in_bf16=up, wpack_bf16=pack(lib, wt.to(dev), 0, 16), bias=bias16, out_nchw=out, c_real=Cs,
                                B=B, H=H, W=W, n_out=16))
        assert rel_l2(out.cpu(), F.conv2d(u, wt, bt, padding=1)) < 2e-3
        # tail dgrad (planar gradient -> 64-feature PTL) and tail wgrad
        dout = torch.randn(B, Cs, H, W)
        d16 = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
        d32 = torch.zeros(rows, 64, device=dev)
        L.check(lib.sres_conv3x3_small_in(ptr(dout.to(dev)), ptr(wt.to(dev)), None, B, Cs, H, W, 1, 0, ptr(d32), ptr(d16),
                                          L.cur_stream()), "tail dgrad")
        torch.cuda.synchronize()
        assert rel_l2(from_ptl(d32, B, H, W).cpu(), F.conv_transpose2d(dout, wt, None, padding=1)) < 1e-5
        dwt = torch.empty(Cs, 64, 3, 3, device=dev)
        dbt = torch.empty(Cs, device=dev)
        L.check(lib.sres_small_out_wgrad(ptr(dout.to(dev)), ptr(up), B, Cs, H, W, ptr(dwt), ptr(dbt), 0, ptr(ws),
                                         C.c_size_t(wsb), L.cur_stream()), "tail wgrad")
        torch.cuda.synchronize()
        assert rel_l2(dwt.cpu(), torch.nn.grad.conv2d_weight(u, (Cs, 64, 3, 3), dout, padding=1)) < 1e-4
        assert rel_l2(dbt.cpu(), dout.sum((0, 2, 3))) < 1e-4


def test_tail_conv_cuda_core_path_and_wide_images(env):
    """64 -> Cs tail conv on CUDA cores (the path for images wider than the tensor-core halo window) and the
    support predicate that selects it."""
    L, lib, dev = env
    # the narrow three-taps-per-MMA kernel stages one 128-row block per kernel row, whatever the image width
    assert lib.sres_conv_supported(192, 192, 16) == 1 and lib.sres_conv_supported(768, 768, 16) == 1
    assert lib.sres_conv_supported(48, 48, 64) == 1 and lib.sres_conv_supported(384, 384, 64) == 1
    for Cs, B, H, W in [(2, 2, 20, 24), (4, 1, 9, 130)]:
        u = bf16_round(torch.randn(B, 64, H, W))
        wt, bt = torch.randn(Cs, 64, 3, 3) * 0.05, torch.randn(Cs)
        out = torch.full((B, Cs, H, W), float("nan"), device=dev)
        L.check(lib.sres_conv3x3_small_out(ptr(to_ptl(u.to(dev), torch.bfloat16)), ptr(wt.to(dev)), ptr(bt.to(dev)), B, Cs, H, W,
                                           ptr(out), L.cur_stream()), "small_out")
        torch.cuda.synchronize()
        assert rel_l2(out.cpu(), F.conv2d(u, wt, bt, padding=1)) < 1e-5


@pytest.mark.parametrize("Cs,B,H,W", [(2, 3, 20, 24), (1, 2, 9, 9), (4, 1, 16, 12), (2, 2, 192, 192), (4, 1, 24, 768), (3, 1, 100, 130)])
def test_tail_conv_tensor_cores_any_width(env, Cs, B, H, W):
    """Tail conv 64 -> Cs on the tensor cores: the narrow (N = 48) three-taps-per-MMA kernel (default; union halo window
    for narrow images, one 128-row block per kernel row for wide ones -- 768-pixel rows of BASELINE config 5 included)
    against fp32 torch on the same bf16 operands, and against the tap-per-MMA N = 16 kernel where that one fits."""
    L, lib, dev = env
    u = bf16_round(torch.randn(B, 64, H, W))
    wt, bt = bf16_round(torch.randn(Cs, 64, 3, 3) * 0.05), torch.randn(Cs)
    ref = F.conv2d(u, wt, bt, padding=1)
    up = to_ptl(u.to(dev), torch.bfloat16)
    bias16 = torch.zeros(16, device=dev)
    bias16[:Cs] = bt.to(dev)
    wp = pack(lib, wt.to(dev), 0, 16)
    out = torch.full((B, Cs, H, W), float("nan"), device=dev)
    run_conv(lib, conv_args(in_bf16=up, wpack_bf16=wp, bias=bias16, out_nchw=out, c_real=Cs, B=B, H=H, W=W, n_out=16))
    assert torch.isfinite(out).all() and rel_l2(out.cpu(), ref) < 2e-3
    if W <= 400:
        old = torch.full((B, Cs, H, W), float("nan"), device=dev)
        run_conv(lib, conv_args(in_bf16=up, wpack_bf16=wp, bias=bias16, out_nchw=old, c_real=Cs, B=B, H=H, W=W, n_out=16,
                                debug_flags=64))
        assert rel_l2(out.cpu(), old.cpu()) < 1e-5


@pytest.mark.parametrize("B,H,W,red", [(3, 20, 24, 2), (2, 48, 48, 16), (4, 7, 9, 4)])
def test_channel_attention_forward_backward(env, B, H, W, red):
    """CALayer + RCAB residual against autograd of the oracle's ca_layer (network.py:44-47, 61-64)."""
    L, lib, dev = env
    hid = 64 // red
    t2 = bf16_round(torch.randn(B, 64, H, W)).requires_grad_(True)
    x = torch.randn(B, 64, H, W)
    sd = {"ca.conv_du.0.weight": (torch.randn(hid, 64, 1, 1) * 0.3).requires_grad_(True), "ca.conv_du.0.bias": torch.randn(hid).requires_grad_(True),
          "ca.conv_du.2.weight": (torch.randn(64, hid, 1, 1) * 0.3).requires_grad_(True), "ca.conv_du.2.bias": torch.randn(64).requires_grad_(True)}
    out_ref = O.ca_layer(t2, sd, "ca") + x
    g = torch.randn(B, 64, H, W)
    out_ref.backward(g)
    w1, b1, w2, b2 = [sd[k].detach().reshape(sd[k].shape[0], -1).contiguous().to(dev) for k in sd]
    t2p = to_ptl(t2.detach().to(dev), torch.bfloat16)
    rows = t2p.shape[0]
    pool_sum = torch.empty(B, 64, device=dev)
    L.check(lib.sres_ca_pool(ptr(t2p), ptr(pool_sum), B, H, W, L.cur_stream()), "ca_pool")
    xo = torch.full((rows, 64), float("nan"), device=dev)
    xb = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
    mean, sv = torch.empty(B, 64, device=dev), torch.empty(B, 64, device=dev)
    L.check(lib.sres_ca_apply_fwd(ptr(t2p), None, ptr(pool_sum), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid,
                                  ptr(to_ptl(x.to(dev), torch.float32)), ptr(xo), ptr(xb), ptr(mean), ptr(sv), B, H, W,
                                  L.cur_stream()), "ca_apply_fwd")
    torch.cuda.synchronize()
    assert rel_l2(from_ptl(xo, B, H, W).cpu(), out_ref.detach()) < 1e-5 and pads_are_zero(xo, B, H, W)
    assert rel_l2(mean.cpu(), t2.detach().mean((2, 3))) < 1e-5
    bpi = lib.sres_ca_blocks_per_image(B, H, W)
    ds_part = torch.empty(B * bpi * 64, device=dev)
    dt2 = torch.full((rows, 64), 7.0, device=dev, dtype=torch.bfloat16)
    ds = torch.empty(B, 64, device=dev)
    L.check(lib.sres_ca_bwd(ptr(to_ptl(g.to(dev), torch.float32)), ptr(t2p), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid,
                            ptr(mean), ptr(ds_part), ptr(dt2), ptr(ds), B, H, W, L.cur_stream()), "ca_bwd")
    torch.cuda.synchronize()
    assert rel_l2(from_ptl(dt2, B, H, W).cpu(), t2.grad) < 6e-3 and pads_are_zero(dt2, B, H, W)
    # parameter gradients: one "layer" laid out as [w1,b1,w2,b2]
    flat = torch.cat([w1.flatten(), b1.flatten(), w2.flatten(), b2.flatten()])
    gflat = torch.full_like(flat, float("nan"))
    lib.sres_ca_param_grads_scratch_bytes.restype = C.c_size_t
    scr = torch.empty(lib.sres_ca_param_grads_scratch_bytes(1, B), dtype=torch.uint8, device=dev)
    L.check(lib.sres_ca_param_grads(ptr(flat), ptr(gflat), C.c_int64(flat.numel()), 1, ptr(mean), ptr(ds), B, hid, 0,
                                    ptr(scr), C.c_size_t(scr.numel()), L.cur_stream()), "ca_param_grads")
    torch.cuda.synchronize()
    ref_flat = torch.cat([sd[k].grad.flatten() for k in sd])
    assert rel_l2(gflat.cpu(), ref_flat) < 1e-4


def test_bicubic_matches_interpolate(env):
    L, lib, dev = env
    from sres_b200 import nn as snn
    for shape, s in [((3, 2, 192, 192), 4), ((2, 1, 20, 28), 2), ((1, 4, 64, 64), 8), ((2, 2, 27, 27), 3)]:
        x = torch.randn(*shape)
        down = snn.bicubic_resize(x.to(dev), 1.0 / s)
        ref = O.downsample(x, s)
        assert down.shape == ref.shape and (down.cpu() - ref).abs().max() < 2e-6
        up = snn.bicubic_resize(down, s)
        assert (up.cpu() - O.upsample(ref, s)).abs().max() < 5e-6


@pytest.mark.parametrize("kind", ["l2", "charbonnier", "l1"])
def test_losses_and_gradients(env, kind):
    L, lib, dev = env
    from sres_b200 import nn as snn
    prd = torch.randn(3, 2, 40, 40, requires_grad=True)
    tar = torch.randn(3, 2, 44, 42)                                  # larger target: conform_to_product crops it
    ref = O.single_product_loss(prd, tar, kind)
    (ref * 1.7).backward()
    p = prd.detach().to(dev).requires_grad_(True)
    got = snn.loss(p, tar.to(dev), kind)
    (got * 1.7).backward()
    assert abs(got.item() - ref.item()) < 1e-6 * max(1.0, abs(ref.item()))
    assert rel_l2(p.grad.cpu(), prd.grad) < 1e-5


def test_fused_adam_matches_torch_adam(env):
    L, lib, dev = env
    n = 4 * 1001
    p0, steps = torch.randn(n), 5
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=3e-3, weight_decay=0.01)
    p, m, v = p0.to(dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    for t in range(1, steps + 1):
        g = torch.randn(n) * (0.1 if t % 2 else 1e-6)
        ref.grad = g.clone()
        opt.step()
        L.check(lib.sres_adam_step_flat(ptr(p), ptr(g.to(dev)), ptr(m), ptr(v), C.c_int64(n), C.c_int64(t), C.c_double(3e-3),
                                        C.c_double(0.9), C.c_double(0.999), C.c_double(1e-8), C.c_double(0.01), L.cur_stream()), "adam")
    torch.cuda.synchronize()
    assert (p.cpu() - ref.detach()).abs().max() < 1e-5
