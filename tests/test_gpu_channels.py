"""5 to 16 image channels through RCAN and EDSR.

The narrow convolutions at the two ends of the network (small_conv.cu) take Cs = 1..16: the weight gradients and the
CUDA-core tail forward run as chunks of <= 4 channels through the 1..4-channel kernels, the head forward and the tail
input-gradient (which sum over the channels) through a kernel of their own for 5..16.  Checked here:

  * without a GPU: the network description accepts 1..16 channels for RCAN and EDSR, refuses 17, and its parameter count
    equals the reference's state_dict;
  * kernel by kernel, against float64 references, at geometries that reach every code path (vector and scalar paths, one
    and several column strips, the three PTL row mappings of the tail input-gradient, accumulate = 1), with every output
    pre-filled with NaN so that an element the kernel should write and does not, or writes and should not, is caught;
  * the whole model against the oracle (training and inference, one fused Adam step), and the controller end to end with
    six variables.
"""
import ctypes as C
import random
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rcan_oracle as O

TOL = 1e-2                        # global rel-L2 of output and gradient against the oracle (BASELINE.json north_star)
TOL_TENSOR = 2e-2                 # head / tail weights and biases, tensor by tensor
WGRAD_REL = 1e-4                  # head / tail weight gradients (fp32), as test_gpu_kernels.test_head_and_tail_convs
CONV_REL = 1e-5                   # head forward / tail input-gradient / CUDA-core tail forward (fp32 out)
CHANNELS = [5, 8, 13, 16]


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU: the network description
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from sres_b200 import _lib as L
    lb = L.lib()
    lb.sres_rcan_param_count.restype = C.c_int64
    lb.sres_last_error.restype = C.c_char_p
    return lb


def _desc(arch, cin, cout):
    from sres_b200.engine import ARCH_EDSR, RcanDesc
    d = RcanDesc()
    d.B, d.H, d.W, d.cin, d.cout, d.nfeatures, d.reduction, d.n_up = 4, 48, 48, cin, cout, 64, 16, 2
    d.up_factor[0] = d.up_factor[1] = 2
    if arch == "edsr":
        d.arch, d.res_scale, d.n_groups, d.n_blocks = ARCH_EDSR, 1.0, 1, 16
        cfg = O.model_cfg(name="edsr")
    else:
        d.n_groups, d.n_blocks = 10, 20
        cfg = O.model_cfg(cbottleneck=16)
    return d, cfg


@pytest.mark.parametrize("arch", ["rcan", "edsr"])
@pytest.mark.parametrize("cin,cout", [(5, 5), (8, 8), (16, 16), (5, 16), (16, 1), (6, 2)])
def test_network_accepts_up_to_16_channels(lib, arch, cin, cout):
    d, cfg = _desc(arch, cin, cout)
    n = lib.sres_rcan_param_count(C.byref(d))
    assert n == sum(int(np.prod(s)) for s in O.param_shapes(cfg, cin, cout).values())
    for training in (0, 1):
        ws = C.c_size_t()
        assert lib.sres_rcan_workspace_bytes(C.byref(d), training, C.byref(ws)) == 0 and ws.value > 0


@pytest.mark.parametrize("arch", ["rcan", "edsr"])
@pytest.mark.parametrize("cin,cout", [(17, 2), (2, 17), (17, 17), (0, 2)])
def test_network_refuses_more_than_16_channels(lib, arch, cin, cout):
    d, _ = _desc(arch, cin, cout)
    assert lib.sres_rcan_param_count(C.byref(d)) < 0
    ws = C.c_size_t()
    assert lib.sres_rcan_workspace_bytes(C.byref(d), 1, C.byref(ws)) == 2          # SRES_ERR_UNSUPPORTED
    assert b"channels" in lib.sres_last_error()


def test_narrow_kernels_refuse_17_channels(lib):
    """The argument checks come before any device work (the pointers are never dereferenced)."""
    p = C.c_void_p(16)
    assert lib.sres_conv3x3_small_in(p, p, None, 1, 17, 8, 8, 0, 0, p, None, None) == 2
    assert b"1..16" in lib.sres_last_error()
    assert lib.sres_conv3x3_small_out(p, p, None, 1, 17, 8, 8, p, None) == 2
    assert lib.sres_small_in_wgrad(p, None, p, 1, 17, 8, 8, p, None, 0, p, C.c_size_t(1 << 30), None) == 2
    assert lib.sres_small_out_wgrad(p, p, 1, 17, 8, 8, p, None, 0, p, C.c_size_t(1 << 30), None) == 2
    assert b"1..16" in lib.sres_last_error()


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU), against float64
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    from sres_b200 import _lib as L
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lb = L.lib()
    lb.sres_small_wgrad_workspace_bytes.restype = C.c_size_t
    return L, lb, torch.device("cuda:0")


def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def _ptl_index(B, H, W, f):
    """Row of every padded position (b, y, x), y <= H, x <= W, in the plain PTL (f = 1) or in the sub-grid-major
    PixelUnshuffle(f) layout the tail input-gradient writes; and the total number of rows of that buffer."""
    b = torch.arange(B).view(B, 1, 1)
    y = torch.arange(H + 1).view(1, H + 1, 1)
    x = torch.arange(W + 1).view(1, 1, W + 1)
    if f == 1:
        return (b * (H + 1) + y) * (W + 1) + x, B * (H + 1) * (W + 1)
    Rl, Pl = H // f + 1, W // f + 1
    sub = (y % f) * f + x % f
    return ((sub * B + b) * Rl + y // f) * Pl + x // f, f * f * B * Rl * Pl


def _expected_rows(ref, f):
    """ref (B, 64, H, W) -> the [rows][64] buffer a kernel writes: values at image positions, zeros at the padding
    positions it owns, NaN wherever it must not write."""
    B, _, H, W = ref.shape
    idx, rows = _ptl_index(B, H, W, f)
    full = torch.zeros(B, H + 1, W + 1, 64, dtype=torch.float64)
    full[:, :H, :W] = ref.permute(0, 2, 3, 1)
    out = torch.full((rows, 64), float("nan"), dtype=torch.float64)
    out[idx.reshape(-1)] = full.reshape(-1, 64)
    return out


def _check_rows(name, got32, got16, exp):
    written = ~torch.isnan(exp[:, 0])
    if got32 is not None:
        g = got32.cpu().double()
        assert torch.isnan(g[~written]).all(), f"{name}: fp32 rows written outside the image and its padding"
        assert torch.isfinite(g[written]).all(), f"{name}: fp32 rows left unwritten"
        e = exp[written]
        rel = ((g[written] - e).norm() / e.norm()).item()
        assert rel < CONV_REL, f"{name}: fp32 rel-L2 {rel:.3e}"
        assert (g[written][e == 0] == 0).all(), f"{name}: padding rows not zero"
    if got16 is not None:
        g = got16.cpu().double()
        assert torch.isnan(g[~written]).all(), f"{name}: bf16 rows written outside the image and its padding"
        e = exp[written]
        e16 = e.float().bfloat16().double()
        gw = g[written]
        assert torch.isfinite(gw).all(), f"{name}: bf16 rows left unwritten"
        # the kernel rounds its fp32 sum once: within one bf16 step of the rounded reference
        # (plus a little slack for sums that cancel to almost zero, where the fp32 rounding is not small relative to them)
        slack = 1e-6 * e.abs().max()
        assert ((gw - e16).abs() <= 2.0 ** -7 * e.abs() + slack).all(), f"{name}: bf16 output off by more than one step"
        assert ((gw - e16).norm() / e16.norm()).item() < 4e-3


# (B, H, W): W % 4 == 0 in one strip / several strips (W > 256), W % 4 != 0 in one strip / several strips
GEOMS_IN = [(2, 20, 24), (1, 16, 768), (2, 9, 13), (1, 6, 514)]


@pytest.mark.gpu
@pytest.mark.parametrize("Cs", CHANNELS)
@pytest.mark.parametrize("B,H,W", GEOMS_IN)
def test_head_conv_forward(env, Cs, B, H, W):
    """sres_conv3x3_small_in, transposed = 0 (head conv Cs -> 64 + bias), fp32 and bf16 PTL outputs."""
    L, lib, dev = env
    g = _gen("head", Cs, B, H, W)
    x = torch.randn(B, Cs, H, W, generator=g)
    w = torch.randn(64, Cs, 3, 3, generator=g) * 0.2
    b = torch.randn(64, generator=g)
    ref = F.conv2d(x.double(), w.double(), b.double(), padding=1)
    rows = B * (H + 1) * (W + 1)
    o32 = torch.full((rows, 64), float("nan"), device=dev)
    o16 = torch.full((rows, 64), float("nan"), device=dev, dtype=torch.bfloat16)
    xd, wd, bd = x.to(dev), w.to(dev), b.to(dev)
    L.check(lib.sres_conv3x3_small_in(L.ptr(xd), L.ptr(wd), L.ptr(bd), B, Cs, H, W, 0, 0, L.ptr(o32), L.ptr(o16),
                                      L.cur_stream()), "head conv")
    torch.cuda.synchronize()
    _check_rows(f"head {Cs} {(B, H, W)}", o32, o16, _expected_rows(ref, 1))


# (unshuffle, B, H, W): plain rows (fp32 + bf16, as the network's x1 tail), PixelUnshuffle(2) / (3) rows (bf16, as the
# x4 / x3 tails), each on the vector path (W % 4 == 0) and the scalar one
GEOMS_DGRAD = [(0, 2, 20, 24), (0, 1, 16, 768), (0, 2, 9, 13),
               (2, 2, 24, 48), (2, 1, 16, 520), (2, 1, 10, 14),
               (3, 2, 18, 36), (3, 1, 9, 15)]


@pytest.mark.gpu
@pytest.mark.parametrize("Cs", CHANNELS)
@pytest.mark.parametrize("f,B,H,W", GEOMS_DGRAD)
def test_tail_input_gradient(env, Cs, f, B, H, W):
    """sres_conv3x3_small_in, transposed = 1 (input-gradient of the tail conv 64 -> Cs: transposed, flipped weights),
    with the plain and the PixelUnshuffle(f) row mappings; every sub-grid compared with the reference's slice."""
    L, lib, dev = env
    g = _gen("dgrad", Cs, f, B, H, W)
    dout = torch.randn(B, Cs, H, W, generator=g)
    wt = torch.randn(Cs, 64, 3, 3, generator=g) * 0.05
    ref = F.conv_transpose2d(dout.double(), wt.double(), None, padding=1)
    _, rows = _ptl_index(B, H, W, max(f, 1))
    o32 = torch.full((rows, 64), float("nan"), device=dev)
    o16 = torch.full((rows, 64), float("nan"), device=dev, dtype=torch.bfloat16)
    dd, wd = dout.to(dev), wt.to(dev)
    L.check(lib.sres_conv3x3_small_in(L.ptr(dd), L.ptr(wd), None, B, Cs, H, W, 1, f, L.ptr(o32), L.ptr(o16),
                                      L.cur_stream()), "tail dgrad")
    torch.cuda.synchronize()
    _check_rows(f"tail dgrad {Cs} f={f} {(B, H, W)}", o32, o16, _expected_rows(ref, max(f, 1)))
    if f > 1:   # the network's call: bf16 only
        o16b = torch.full((rows, 64), float("nan"), device=dev, dtype=torch.bfloat16)
        L.check(lib.sres_conv3x3_small_in(L.ptr(dd), L.ptr(wd), None, B, Cs, H, W, 1, f, None, L.ptr(o16b),
                                          L.cur_stream()), "tail dgrad (bf16 only)")
        torch.cuda.synchronize()
        assert torch.equal(o16b.view(torch.int16), o16.view(torch.int16))


def _wgrad_ref(x, dy):
    """float64 weight gradient of a 3x3, padding-1 conv: x (B,Ci,H,W), dy (B,Co,H,W) -> (Co,Ci,3,3)."""
    return torch.nn.grad.conv2d_weight(x.double(), (dy.shape[1], x.shape[1], 3, 3), dy.double(), padding=1)


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm()).item()


GEOMS_WG = [(2, 20, 24), (1, 16, 768), (2, 9, 13)]


@pytest.mark.gpu
@pytest.mark.parametrize("Cs", CHANNELS)
@pytest.mark.parametrize("B,H,W", GEOMS_WG)
def test_head_weight_gradient(env, Cs, B, H, W):
    """sres_small_in_wgrad (head conv Cs -> 64) from two fp32 PTL gradient addends; then g2 = NULL, accumulate = 1,
    db = NULL: dw grows by the g1 gradient and db keeps its value bit for bit."""
    from gpu_util import to_ptl
    L, lib, dev = env
    g = _gen("head wgrad", Cs, B, H, W)
    x = torch.randn(B, Cs, H, W, generator=g)
    g1, g2 = torch.randn(B, 64, H, W, generator=g), torch.randn(B, 64, H, W, generator=g)
    xd = x.to(dev)
    g1p, g2p = to_ptl(g1.to(dev), torch.float32), to_ptl(g2.to(dev), torch.float32)
    wsb = lib.sres_small_wgrad_workspace_bytes()
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    dw = torch.full((64, Cs, 3, 3), float("nan"), device=dev)
    db = torch.full((64,), float("nan"), device=dev)
    L.check(lib.sres_small_in_wgrad(L.ptr(g1p), L.ptr(g2p), L.ptr(xd), B, Cs, H, W, L.ptr(dw), L.ptr(db), 0, L.ptr(ws),
                                    C.c_size_t(wsb), L.cur_stream()), "head wgrad")
    torch.cuda.synchronize()
    gs = g1.double() + g2.double()
    assert torch.isfinite(dw).all() and torch.isfinite(db).all()
    assert _rel(dw, _wgrad_ref(x, gs)) < WGRAD_REL
    assert _rel(db, gs.sum((0, 2, 3))) < WGRAD_REL
    dw1, db1 = dw.clone(), db.clone()
    L.check(lib.sres_small_in_wgrad(L.ptr(g1p), None, L.ptr(xd), B, Cs, H, W, L.ptr(dw), None, 1, L.ptr(ws),
                                    C.c_size_t(wsb), L.cur_stream()), "head wgrad, accumulate")
    torch.cuda.synchronize()
    assert _rel(dw, dw1.double().cpu() + _wgrad_ref(x, g1)) < WGRAD_REL
    assert torch.equal(db, db1), "db = NULL must leave the bias gradient alone"


@pytest.mark.gpu
@pytest.mark.parametrize("Cs", CHANNELS + [7, 11])     # 7, 11: a remainder of three channels runs as 2 + 1
@pytest.mark.parametrize("B,H,W", GEOMS_WG)
def test_tail_weight_gradient(env, Cs, B, H, W):
    """sres_small_out_wgrad (tail conv 64 -> Cs) from the planar fp32 output gradient and the bf16 PTL conv input; then
    accumulate = 1 with db = NULL: dw doubles and db keeps its value bit for bit."""
    from gpu_util import to_ptl
    L, lib, dev = env
    g = _gen("tail wgrad", Cs, B, H, W)
    u = torch.randn(B, 64, H, W, generator=g).bfloat16().float()
    dout = torch.randn(B, Cs, H, W, generator=g)
    up, dd = to_ptl(u.to(dev), torch.bfloat16), dout.to(dev)
    wsb = lib.sres_small_wgrad_workspace_bytes()
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    dw = torch.full((Cs, 64, 3, 3), float("nan"), device=dev)
    db = torch.full((Cs,), float("nan"), device=dev)
    L.check(lib.sres_small_out_wgrad(L.ptr(dd), L.ptr(up), B, Cs, H, W, L.ptr(dw), L.ptr(db), 0, L.ptr(ws),
                                     C.c_size_t(wsb), L.cur_stream()), "tail wgrad")
    torch.cuda.synchronize()
    ref = _wgrad_ref(u, dout)
    assert torch.isfinite(dw).all() and torch.isfinite(db).all()
    assert _rel(dw, ref) < WGRAD_REL
    assert _rel(db, dout.double().sum((0, 2, 3))) < WGRAD_REL
    db1 = db.clone()
    L.check(lib.sres_small_out_wgrad(L.ptr(dd), L.ptr(up), B, Cs, H, W, L.ptr(dw), None, 1, L.ptr(ws),
                                     C.c_size_t(wsb), L.cur_stream()), "tail wgrad, accumulate")
    torch.cuda.synchronize()
    assert _rel(dw, 2 * ref) < WGRAD_REL
    assert torch.equal(db, db1), "db = NULL must leave the bias gradient alone"


@pytest.mark.gpu
@pytest.mark.parametrize("Cs", CHANNELS)
@pytest.mark.parametrize("B,H,W", [(2, 9, 13), (1, 8, 130)])
def test_tail_conv_cuda_cores(env, Cs, B, H, W):
    """sres_conv3x3_small_out: the CUDA-core tail forward 64 -> Cs, written plane chunk by plane chunk."""
    from gpu_util import to_ptl
    L, lib, dev = env
    g = _gen("tail fwd", Cs, B, H, W)
    u = torch.randn(B, 64, H, W, generator=g).bfloat16().float()
    wt, bt = torch.randn(Cs, 64, 3, 3, generator=g) * 0.05, torch.randn(Cs, generator=g)
    up, wd, bd = to_ptl(u.to(dev), torch.bfloat16), wt.to(dev), bt.to(dev)
    out = torch.full((B, Cs, H, W), float("nan"), device=dev)
    L.check(lib.sres_conv3x3_small_out(L.ptr(up), L.ptr(wd), L.ptr(bd), B, Cs, H, W, L.ptr(out), L.cur_stream()),
            "tail fwd")
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    assert _rel(out, F.conv2d(u.double(), wt.double(), bt.double(), padding=1)) < CONV_REL


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU), against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _build(cfg, cin, cout, dev):
    from sres_b200 import nn as snn
    if O.is_edsr(cfg):
        return snn.EDSR(nchannels_in=cin, nchannels_out=cout, nfeatures=64, nlayers=cfg["nlayers"], scale=O.scale_of(cfg),
                        res_scale=cfg["res_scale"], device=dev)
    return snn.RCAN(nchannels_in=cin, nchannels_out=cout, nfeatures=64, nlayers=cfg["nlayers"], nblocks=cfg["nblocks"],
                    cbottleneck=cfg["cbottleneck"], scale=O.scale_of(cfg), device=dev)


MODEL_CASES = {   # name: (cfg overrides, cin, cout, B, LR tile size)
    "rcan_x4_8ch": (dict(nlayers=2, nblocks=2), 8, 8, 2, 16),
    "rcan_x4_6to2": (dict(nlayers=2, nblocks=2), 6, 2, 2, 16),
    "rcan_x3_16ch": (dict(nlayers=1, nblocks=2, downscale_factors=[3]), 16, 16, 2, 16),
    "edsr_x4_8ch": (dict(name="edsr", nlayers=2), 8, 8, 2, 16),
    "rcan_x8_16ch_wide": (dict(nlayers=1, nblocks=1, downscale_factors=[2, 2, 2]), 16, 16, 1, 96),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_model_matches_oracle(name):
    """Forward + backward against the oracle's autograd (O.forward_backward) on the same LR input and output gradient:
    global rel-L2 of the output and of the full gradient <= 1e-2, head and tail weights / biases <= 2e-2 each; the
    inference-mode forward against the same output; one fused Adam step against the oracle's Adam on the GPU's gradients."""
    from synth import synth_hr
    from sres_b200 import nn as snn
    assert torch.cuda.is_available()
    dev = torch.device("cuda:0")
    over, cin, cout, B, S = MODEL_CASES[name]
    cfg = O.model_cfg(**over)
    scale = O.scale_of(cfg)
    sd = O.make_state_dict(cfg, cin, cout)
    x = O.downsample(synth_hr(B, cin, S * scale, smooth=True), scale).contiguous()
    dout = torch.randn(B, cout, S * scale, S * scale, generator=_gen("dout", name)) * 1e-2
    prd_o, grads_o = O.forward_backward(x, dout, sd, cfg)
    model = _build(cfg, cin, cout, dev)
    assert [k for k, _ in model.named_parameters()] == list(sd.keys())
    model.load_state_dict(sd)
    prd = model(x.to(dev).requires_grad_(True))
    assert prd.shape == (B, cout, S * scale, S * scale)
    prd.backward(dout.to(dev))
    torch.cuda.synchronize()
    ro = _rel(prd.detach(), prd_o)
    params = dict(model.named_parameters())
    num = sum((p.grad.cpu() - grads_o[k]).double().pow(2).sum().item() for k, p in params.items())
    den = sum(g.double().pow(2).sum().item() for g in grads_o.values())
    rg = (num / den) ** 0.5
    ends = {k: _rel(params[k].grad, grads_o[k]) for k in ("head.0.weight", "head.0.bias", "tail.1.weight", "tail.1.bias")}
    print(f"\n  {name}: output rel-L2 {ro:.2e}, gradient rel-L2 {rg:.2e}, " + ", ".join(f"{k} {v:.2e}" for k, v in ends.items()))
    assert ro < TOL and rg < TOL
    for k, v in ends.items():
        assert v < TOL_TENSOR, (k, v)
    # one fused Adam step from the GPU's gradients against the oracle's Adam on the same gradients
    grads_gpu = {k: p.grad.detach().cpu().clone() for k, p in params.items()}
    opt = snn.FusedAdam(model, lr=1e-4)
    opt.step()
    torch.cuda.synchronize()
    sd_ref = {k: v.clone() for k, v in sd.items()}
    adam = O.AdamState(sd_ref, lr=1e-4)
    with torch.no_grad():
        adam.step(sd_ref, grads_gpu)
    for k, p in params.items():
        assert (p.detach().cpu() - sd_ref[k]).abs().max() < 1e-6, k
    # inference mode: the same kernels without saved activations
    model.load_state_dict(sd)
    with torch.no_grad():
        prd2 = model(x.to(dev))
    assert _rel(prd2, prd_o) < TOL


# ---------------------------------------------------------------------------------------------------------------------
# controller level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_controller_six_variables(tmp_path):
    """The reference's workflow with six input and six target variables on the synthetic dataset: two training epochs,
    stitched inference images for every variable, a checkpoint with the reference's state_dict for 6 -> 6 channels."""
    from sres.base.util.config import ConfigContext
    from sres.controller.config import ResultStructure, TSet
    from sres.controller.workflow import WorkflowController
    assert torch.cuda.is_available()
    names = ["SSS", "SST", "SSH", "U", "V", "W"]
    ConfigContext.deactivate()
    random.seed(3)
    wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local"), seed=1)
    wc.initialize("sres", "rcan-10-20-64", **{
        "model.nlayers": 2, "model.nblocks": 2, "task.batch_size": 8, "task.lr": 2e-4, "task.tile_size": dict(x=12, y=12),
        "task.tile_order": "corrected", "dataset.region": dict(ys=480, xs=480), "dataset.ntimes": 4,
        "task.ttsplit": dict(train=0.75, valid=0.25, test=0.0), "platform.results": str(tmp_path),
        "task.input_variables": {n: n.lower() for n in names}, "task.target_variables": list(names)})
    try:
        tr = wc.trainer
        res = tr.train(2, True, seed=4456, interp_loss=True, verbose=False)
        assert np.isfinite(res["prediction"])
        ck = torch.load(tr.checkpoint_manager.checkpoint_path(TSet.Train), map_location="cpu", weights_only=False)
        shapes = O.param_shapes(O.model_cfg(nlayers=2, nblocks=2), 6, 6)
        assert list(ck["model_state_dict"].keys()) == list(shapes.keys())
        assert all(tuple(ck["model_state_dict"][k].shape) == tuple(s) for k, s in shapes.items())
        images, losses = wc.inference(0, ResultStructure.Image)
        assert set(images) == set(names)
        for v in names:
            assert set(images[v]) == {"input", "target", "interpolated", "model"}
            assert images[v]["target"].shape == (480 // 48 * 48, 480 // 48 * 48) and images[v]["input"].shape == (120, 120)
            assert images[v]["model"].shape == images[v]["target"].shape
            assert np.isfinite(losses[v]["model"]) and losses[v]["interpolated"] > 0
    finally:
        ConfigContext.deactivate()
