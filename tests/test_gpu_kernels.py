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
    # fp32 and bf16 outputs in separate calls (together they would not fit the N = 192 kernel's epilogue slabs)
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


@pytest.mark.parametrize("B,H,W", [(3, 20, 24), (5, 48, 48), (2, 96, 96)])
def test_conv_n192_matches_tap_per_mma_kernel(env, B, H, W):
    """The three-taps-per-MMA kernel (N = 192, shifted accumulator sum in the epilogue; debug flag 128 forces it for
    every flavour it supports) against the tap-per-MMA kernel (debug flag 64) for every epilogue flavour: same operands, fp32 accumulation in a
    different order, so fp32 outputs agree to 1e-5 relative and bf16 outputs to one rounding step."""
    L, lib, dev = env
    rows = lib.sres_ptl_rows(B, H, W)
    nt = (rows + 125) // 126       # per-tile partial sums of the forced N = 192 kernel: 126-row tiles
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
        "group tail": dict(bias=bias, o16=True, o32=True, rmw=True),
        "body tail": dict(bias=bias, o16=True, resid=True),
        "plain fp32": dict(o32=True),
    }
    for name, f in flavours.items():
        results = []
        for dbg in (128, 128 | 16, 64):
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
            if f.get("resid"):
                kw["resid_f32"] = trunk
            if f.get("part"):
                kw["pool_part"] = part
            run_conv(lib, conv_args(**kw))
            results.append((out16, out32, image_sums(part, B, H, W, 128 if dbg == 64 else 126)))
            del kw
        ref16, ref32, refp = results[2]
        for out16, out32, psum in results[:2]:
            if f.get("o16"):
                assert torch.isfinite(out16.float()).all() and pads_are_zero(out16, B, H, W), name
                # one bf16 rounding step at most, and only where the fp32 sums straddle a rounding boundary
                d = (out16.float() - ref16.float()).abs()
                assert bool((d <= 2.0 ** -7 * ref16.float().abs() + 1e-5).all()), name
                assert float((d > 0).float().mean()) < 2e-2, name
            if f.get("o32"):
                assert torch.isfinite(out32).all() and pads_are_zero(out32, B, H, W), name
                assert rel_l2(out32.cpu(), ref32.cpu()) < 1e-5, name
            if f.get("part"):
                assert rel_l2(psum, refp) < 1e-5, name
        # the compile-time flavour and the runtime-flag instance of the same kernel are bit-equal
        assert torch.equal(results[0][0].nan_to_num(0.0), results[1][0].nan_to_num(0.0)), name
        assert torch.equal(results[0][1].nan_to_num(0.0), results[1][1].nan_to_num(0.0)), name


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
        a1.debug_flags = a2.debug_flags = 64          # two launches of the tap-per-MMA kernel
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
    """The tap-per-MMA kernel (debug flag 64; wide-image / PixelShuffle paths and the A/B baseline of the N = 192 kernel):
    its compile-time epilogue flavours, their row-layout variant (+32), the generic runtime-flag kernel (+16) and the
    opt-in CTA-pair kernel (+8) compute the same thing: outputs bit-equal, per-tile partial sums equal up to summation order."""
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
        for dbg in (64, 64 | 32, 64 | 16, 64 | 8):
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


@pytest.mark.parametrize("n128", ["0", "1"])
@pytest.mark.parametrize("B,H,W", GEOMS[:4])
def test_conv_wgrad(env, B, H, W, n128, monkeypatch):
    """One-job weight gradient against fp64 on the same bf16 operands: products are exact in fp32, only the summation order
    differs.  Bounds at ~10x the rel-L2 measured on a B200 (dw <= 2.5e-7, db <= 1.7e-7), every element within 2^-12 of its |x||dy| sum."""
    monkeypatch.setenv("SRES_WGRAD_N128", n128)   # plain two-taps-per-MMA scheme and the opt-in four-taps one
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


@pytest.mark.parametrize("B,H,W,red", [(3, 20, 24, 2), (2, 48, 48, 16)])
def test_channel_attention_split_trunk_equals_fp32_trunk(env, B, H, W, red):
    """sres_ca_apply_fwd_split (trunk as a bf16 pair hi + lo) against sres_ca_apply_fwd (fp32 trunk), two chained RCAB
    residual updates (network.py:61-64): hi is bit-for-bit the fp32 kernel's bf16 copy of the same input, hi + lo is the
    fp32 value to 2^-17, and both stay zero on the padding rows."""
    L, lib, dev = env
    hid = 64 // red
    w1, b1 = (torch.randn(hid, 64) * 0.3).to(dev), torch.randn(hid).to(dev)
    w2, b2 = (torch.randn(64, hid) * 0.3).to(dev), torch.randn(64).to(dev)
    x0 = to_ptl((torch.randn(B, 64, H, W) * 3).to(dev), torch.float32)
    rows = x0.shape[0]
    mean, sv = torch.empty(B, 64, device=dev), torch.empty(B, 64, device=dev)
    mean2, sv2 = torch.empty(B, 64, device=dev), torch.empty(B, 64, device=dev)
    pool_sum = torch.empty(B, 64, device=dev)
    st = L.cur_stream()
    x_f32 = x0                      # fp32 trunk fed to the fp32 kernel
    hi = lo = None
    for step in range(2):
        t2p = to_ptl(bf16_round(torch.randn(B, 64, H, W)).to(dev), torch.bfloat16)
        L.check(lib.sres_ca_pool(ptr(t2p), ptr(pool_sum), B, H, W, st), "ca_pool")
        xin = x_f32 if step == 0 else (hi.float() + lo.float())    # the value the pair represents (before lo is overwritten)
        hi_out = torch.full((rows, 64), 7.0, device=dev, dtype=torch.bfloat16)
        lo_out = lo if lo is not None else torch.full((rows, 64), 7.0, device=dev, dtype=torch.bfloat16)   # in place from step 1 on
        L.check(lib.sres_ca_apply_fwd_split(ptr(t2p), None, ptr(pool_sum), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid,
                                            ptr(x0) if step == 0 else None, None if step == 0 else ptr(hi), None if step == 0 else ptr(lo),
                                            ptr(hi_out), ptr(lo_out), ptr(mean), ptr(sv), B, H, W, st), "ca_apply_fwd_split")
        # the fp32 kernel on the same value
        xo = torch.full((rows, 64), float("nan"), device=dev)
        xb = torch.zeros(rows, 64, device=dev, dtype=torch.bfloat16)
        L.check(lib.sres_ca_apply_fwd(ptr(t2p), None, ptr(pool_sum), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid, ptr(xin), ptr(xo), ptr(xb),
                                      ptr(mean2), ptr(sv2), B, H, W, st), "ca_apply_fwd")
        torch.cuda.synchronize()
        assert torch.equal(hi_out.view(torch.int16), xb.view(torch.int16))
        assert torch.equal(mean, mean2) and torch.equal(sv, sv2)
        pair = hi_out.float() + lo_out.float()
        err = (pair - xo).abs()
        assert bool((err <= xo.abs() * 2.0 ** -17 + 1e-30).all()), float((err / (xo.abs() + 1e-30)).max())
        assert pads_are_zero(hi_out, B, H, W) and pads_are_zero(lo_out, B, H, W)
        hi, lo = hi_out, lo_out
    # argument errors are reported, not guessed around
    assert lib.sres_ca_apply_fwd_split(ptr(t2p), None, ptr(pool_sum), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid, ptr(x0), ptr(hi), ptr(lo),
                                       ptr(hi_out), ptr(lo_out), ptr(mean), ptr(sv), B, H, W, st) != 0
    assert lib.sres_ca_apply_fwd_split(ptr(t2p), None, ptr(pool_sum), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid, None, ptr(hi), None,
                                       ptr(hi_out), ptr(lo_out), ptr(mean), ptr(sv), B, H, W, st) != 0


@pytest.mark.parametrize("B,H,W,nb,red,training", [(3, 20, 24, 3, 4, True), (2, 48, 48, 2, 16, True), (5, 12, 12, 2, 16, False),
                                                   (2, 48, 48, 3, 16, False), (1, 9, 9, 2, 2, True)])
def test_rcab_chain_equals_kernel_by_kernel(env, B, H, W, nb, red, training):
    """sres_rcab_chain_fwd (a residual group's RCABs in one image-resident cluster launch, network.py:50-77) against the same
    blocks run kernel by kernel (two convolution launches, sres_ca_pool, sres_ca_apply_fwd): the first block's T1 / T2 are
    bit-identical (same MMA order per output row); the pooled mean is summed in another order, so from the gate on the two
    paths agree to fp32 round-off (plus a rare bf16 rounding flip downstream)."""
    L, lib, dev = env
    if not lib.sres_rcab_chain_supported(B, H, W):
        pytest.skip("geometry not served by the chain kernel")
    hid = 64 // red
    RP = (H + 1) * (W + 1)
    rows = B * RP
    KW = 64 * 64 * 9
    stride = 2 * (KW + 64) + hid * 64 + hid + 64 * hid + 64
    g = torch.Generator().manual_seed(B * 1000 + H * 10 + nb)
    params = torch.empty(nb, stride)
    for r in range(nb):
        params[r] = torch.cat([(torch.randn(KW, generator=g) * 0.04), torch.randn(64, generator=g) * 0.1,
                               (torch.randn(KW, generator=g) * 0.04), torch.randn(64, generator=g) * 0.1,
                               torch.randn(hid * 64, generator=g) * 0.3, torch.randn(hid, generator=g),
                               torch.randn(64 * hid, generator=g) * 0.3, torch.randn(64, generator=g)])
    params = params.to(dev).contiguous()
    wpack = torch.empty(nb * 2, KW, device=dev, dtype=torch.bfloat16)
    for r in range(nb):
        for c in range(2):
            w = params[r, c * (KW + 64): c * (KW + 64) + KW].reshape(64, 64, 3, 3).contiguous()
            wpack[2 * r + c] = pack(lib, w, 0)
    x0 = to_ptl(torch.randn(B, 64, H, W, generator=g).to(dev), torch.float32)
    st = L.cur_stream()
    n_xb, n_t = (nb + 2, nb) if training else (2, 1)
    xb_first = 1 if training else 0

    def fresh():
        xb = torch.full((n_xb, rows, 64), 7.0, device=dev, dtype=torch.bfloat16)
        xb[xb_first] = x0.bfloat16()
        return (xb, torch.full((n_t, rows, 64), 7.0, device=dev, dtype=torch.bfloat16), torch.full((n_t, rows, 64), 7.0, device=dev, dtype=torch.bfloat16),
                torch.full((rows, 64), float("nan"), device=dev), torch.zeros(nb if training else 1, B, 64, device=dev), torch.zeros(nb if training else 1, B, 64, device=dev))

    # ---- kernel by kernel ----
    xb_r, t1_r, t2_r, xf_r, mean_r, s_r = fresh()
    pool_sum = torch.empty(B, 64, device=dev)
    fused_pool = RP >= 128
    pool_part = torch.zeros(lib.sres_conv_mtiles(B, H, W), 2, 4, 64, device=dev)
    tol = 3e-4 * nb if fused_pool else 5e-3    # a 1-ulp difference of a gate flips a few bf16 roundings per block, and those spread
    for r in range(nb):
        xi, xo = ((xb_first + r) % 2, (xb_first + r + 1) % 2) if not training else (xb_first + r, xb_first + r + 1)
        ti, si = (r, r) if training else (0, 0)
        pr = params[r]
        o = 0
        c1b = pr[KW:KW + 64]; c2b = pr[2 * KW + 64: 2 * KW + 128]
        o = 2 * (KW + 64)
        w1 = pr[o:o + hid * 64]; b1 = pr[o + hid * 64: o + hid * 64 + hid]
        o2 = o + hid * 64 + hid
        w2 = pr[o2:o2 + 64 * hid]; b2 = pr[o2 + 64 * hid: o2 + 64 * hid + 64]
        run_conv(lib, conv_args(in_bf16=xb_r[xi], wpack_bf16=wpack[2 * r], bias=c1b, out_bf16=t1_r[ti], B=B, H=H, W=W, n_out=64, epi_flags=L.EPI_RELU))
        if fused_pool:   # the production path: channel sums of the fp32 accumulators in the conv2 epilogue, like the chain kernel
            run_conv(lib, conv_args(in_bf16=t1_r[ti], wpack_bf16=wpack[2 * r + 1], bias=c2b, out_bf16=t2_r[ti], pool_part=pool_part, B=B, H=H, W=W,
                                    n_out=64, epi_flags=L.EPI_POOL))
        else:            # small images: sres_ca_pool sums the bf16-ROUNDED T2 (means differ by the mean rounding error, ~1e-3 relative)
            run_conv(lib, conv_args(in_bf16=t1_r[ti], wpack_bf16=wpack[2 * r + 1], bias=c2b, out_bf16=t2_r[ti], B=B, H=H, W=W, n_out=64, epi_flags=0))
            L.check(lib.sres_ca_pool(ptr(t2_r[ti]), ptr(pool_sum), B, H, W, st), "ca_pool")
        L.check(lib.sres_ca_apply_fwd(ptr(t2_r[ti]), ptr(pool_part) if fused_pool else None, None if fused_pool else ptr(pool_sum), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid,
                                      ptr(x0 if r == 0 else xf_r), ptr(xf_r), ptr(xb_r[xo]), ptr(mean_r[si]), ptr(s_r[si]), B, H, W, st), "ca_apply_fwd")
    torch.cuda.synchronize()

    # ---- one chain launch ----
    xb_c, t1_c, t2_c, xf_c, mean_c, s_c = fresh()
    scratch = torch.zeros(lib.sres_rcab_chain_scratch_bytes(B) // 4, device=dev)
    a = L.ChainArgs()
    a.xb_bf16, a.t1_bf16, a.t2_bf16 = xb_c.data_ptr(), t1_c.data_ptr(), t2_c.data_ptr()
    a.wpack_bf16, a.params, a.x_in_f32, a.x_f32 = wpack.data_ptr(), params.data_ptr(), x0.data_ptr(), xf_c.data_ptr()
    a.save_mean, a.save_s, a.scratch = mean_c.data_ptr(), s_c.data_ptr(), scratch.data_ptr()
    a.rcab_stride, a.save_stride = stride, (B * 64 if training else 0)
    a.B, a.H, a.W, a.n_blocks, a.hidden = B, H, W, nb, hid
    a.xb_first, a.xb_ring, a.xb_count = xb_first, (0 if training else 2), n_xb
    a.t_first, a.t_fixed, a.t_count = 0, (0 if training else 1), n_t
    L.check(lib.sres_rcab_chain_fwd(C.byref(a), st), "sres_rcab_chain_fwd")
    torch.cuda.synchronize()

    if training:
        assert torch.equal(t1_c[0].view(torch.int16), t1_r[0].view(torch.int16))
        assert torch.equal(t2_c[0].view(torch.int16), t2_r[0].view(torch.int16))
        for r in range(nb):
            assert rel_l2(t1_c[r].float(), t1_r[r].float()) < tol and rel_l2(t2_c[r].float(), t2_r[r].float()) < tol, r
            assert rel_l2(xb_c[xb_first + r + 1].float(), xb_r[xb_first + r + 1].float()) < tol, r
            assert pads_are_zero(t1_c[r], B, H, W) and pads_are_zero(t2_c[r], B, H, W) and pads_are_zero(xb_c[xb_first + r + 1], B, H, W)
        assert torch.equal(xb_c[0], xb_r[0]) and torch.equal(xb_c[xb_first], xb_r[xb_first])     # untouched buffers stay untouched
    else:
        last = (xb_first + nb) % 2
        assert rel_l2(xb_c[last].float(), xb_r[last].float()) < tol and pads_are_zero(xb_c[last], B, H, W)
    assert rel_l2(mean_c, mean_r) < tol and rel_l2(s_c, s_r) < tol
    assert rel_l2(xf_c, xf_r) < tol and pads_are_zero(xf_c, B, H, W)
    # run to run: bit-identical (fixed summation orders, no atomics)
    xb_d, t1_d, t2_d, xf_d, mean_d, s_d = fresh()
    a.xb_bf16, a.t1_bf16, a.t2_bf16, a.x_f32, a.save_mean, a.save_s = xb_d.data_ptr(), t1_d.data_ptr(), t2_d.data_ptr(), xf_d.data_ptr(), mean_d.data_ptr(), s_d.data_ptr()
    L.check(lib.sres_rcab_chain_fwd(C.byref(a), st), "sres_rcab_chain_fwd")
    torch.cuda.synchronize()
    assert torch.equal(xf_d, xf_c) and torch.equal(s_d, s_c) and torch.equal(t2_d.view(torch.int16), t2_c.view(torch.int16))


@pytest.mark.parametrize("setting", ["SRES_CHAIN_OVERLAP=1", "SRES_CHAIN_LEND=1", "SRES_CHAIN_BULK=1", "SRES_CHAIN_K=1", "SRES_CHAIN_LEND=1 SRES_CHAIN_BULK=1"])
def test_rcab_chain_variants_keep_parity(setting):
    """The chain kernel's measured variants (streaming under the next conv1 with six extra warps, 4-deep halo ring through the
    idle weight region, bulk-copy streaming phase, one CTA per image) are selected by environment switches that the library
    reads once per process: the same kernel-by-kernel parity test runs in a fresh interpreter for each of them."""
    import os
    import subprocess
    import sys
    env_ = dict(os.environ)
    for kv in setting.split():
        key, val = kv.split("=")
        env_[key] = val
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(here, "test_gpu_kernels.py"), "-q", "-x", "-m", "gpu", "-k",
                        "test_rcab_chain_equals_kernel_by_kernel", "-p", "no:cacheprovider"], env=env_, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "5 passed" in r.stdout, r.stdout[-1000:]


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
