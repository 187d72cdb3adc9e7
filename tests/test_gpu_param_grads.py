"""Parameter-gradient kernels, tensor by tensor, against float64 references at the shapes the backward pass calls them with.

An error in an input-gradient kernel flows upstream into every gradient before it, so the model-level tests see it.  An
error in a parameter-gradient kernel lands in one tensor, or one slice of one, and nowhere else: a norm check cannot see
a permuted tap, a permuted output channel or a wrong PixelShuffle sub-convolution offset.  So every check here compares
ONE tensor element by element with plain PyTorch in float64, computed from the operands the kernel reads (bf16-rounded
where it reads bf16), and reports two numbers (visible with `pytest -s`):

    rel-L2      ||got - ref|| / ||ref||  of the tensor (weights and biases separately)
    max|err|/A  worst element error over A, the same reduction taken over |operands|

Products of bf16 operands are exact in fp32, so only the fp32 summation order separates a correct kernel from the
reference.  The rel-L2 bounds sit at about ten times the largest value measured on a B200 (quoted in each docstring),
and every element must be within 2^-12 A.
"""
import ctypes as C
import zlib

import pytest
import torch

from gpu_util import check_grad, conv3x3_wgrad_ref, pads_are_zero, ptr, to_ptl

pytestmark = pytest.mark.gpu

KW = 64 * 64 * 9            # one 64 -> 64 3x3 conv weight
SCALE = float(torch.tensor(0.1, dtype=torch.float32))   # EDSR res_scale as the kernel holds it (fp32)

# rel-L2 bounds: about 10x the largest value measured on a B200 (NVIDIA B200, 1000 W power limit) at the shapes below
WG_CHUNK = 1.5e-6    # sres_conv3x3_wgrad_batch dw, per 128-position chunk a CTA accumulates (see wg_bound)
WG_B = 3e-6          # sres_conv3x3_wgrad_batch db (summed on CUDA cores): measured <= 2.5e-7
SO_W, SO_B = 6e-6, 5e-6     # sres_small_out_wgrad (tail): measured <= 6.0e-7 / 4.8e-7
SI_W, SI_B = 5e-6, 5e-6     # sres_small_in_wgrad (head): measured <= 4.7e-7 / 4.4e-7
CA_P = 7e-6                 # sres_ca_param_grads w1, b1, w2, b2, B > 1: measured <= 6.3e-7
# B = 1: dw2 = dz h^T is a single outer product, so nothing averages out the fp32 rounding of a hidden unit h that
# W1 m + b1 leaves close to zero (its error is relative to |W1||m| + |b1|, not to |h|): measured 4.5e-6 for hid 4
# (every element within 1.2e-8 A), <= 7.6e-7 otherwise
CA_P_B1 = 5e-5
CA_DS = 1e-6                # sres_ca_bwd_apply save_ds: measured <= 9.7e-8


@pytest.fixture(scope="module")
def env():
    from sres_b200 import _lib as L
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = L.lib()
    dev = torch.device("cuda:0")
    print(f"\n  device: {torch.cuda.get_device_name(dev)}")
    lib.sres_conv_wgrad_workspace_bytes.restype = C.c_size_t
    lib.sres_small_wgrad_workspace_bytes.restype = C.c_size_t
    lib.sres_ca_param_grads_scratch_bytes.restype = C.c_size_t
    return L, lib, dev


def _gen(dev, *key):
    return torch.Generator(device=dev).manual_seed(zlib.crc32(repr(key).encode()))


def _bf16(g, dev, *shape):
    return torch.randn(*shape, device=dev, generator=g).bfloat16()


# ---------------------------------------------------------------------------------------------------------------------
# A. sres_conv3x3_wgrad_batch
# ---------------------------------------------------------------------------------------------------------------------
class Job:
    """One weight-gradient job: NCHW bf16 operands (the reference's) and their PTL copies (the kernel's)."""

    def __init__(self, x, dy, dw, db, cout_total=64, stride=1, offset=0, acc=0, scale=1.0):
        self.x, self.dy = x, dy
        self.xp, self.dyp = to_ptl(x, torch.bfloat16), to_ptl(dy, torch.bfloat16)
        self.dw, self.db = dw, db
        self.cout_total, self.stride, self.offset, self.acc, self.scale = cout_total, stride, offset, acc, scale

    def c(self, L):
        return L.WgradJob(self.xp.data_ptr(), self.dyp.data_ptr(), self.dw.data_ptr(),
                          self.db.data_ptr() if self.db is not None else None,
                          self.cout_total, self.stride, self.offset, self.acc, self.scale)


def run_batch(env, jobs, B, H, W, ws, sync=True):
    L, lib, dev = env
    arr = (L.WgradJob * len(jobs))(*[j.c(L) for j in jobs])
    L.check(lib.sres_conv3x3_wgrad_batch(arr, len(jobs), B, H, W, ptr(ws), C.c_size_t(ws.numel()), L.cur_stream()),
            "sres_conv3x3_wgrad_batch")
    if sync:
        torch.cuda.synchronize()


def workspace(env):
    L, lib, dev = env
    return torch.empty(lib.sres_conv_wgrad_workspace_bytes(), dtype=torch.uint8, device=dev)


def plain_jobs(env, B, H, W, n, seed=0):
    dev = env[2]
    g = _gen(dev, "plain", B, H, W, n, seed)
    return [Job(_bf16(g, dev, B, 64, H, W), _bf16(g, dev, B, 64, H, W), torch.full((64, 64, 3, 3), float("nan"), device=dev),
                torch.full((64,), float("nan"), device=dev)) for _ in range(n)]


def wg_bound(env, B, H, W, njobs):
    """rel-L2 bound of a 3x3 weight gradient.  Each CTA accumulates its share of a job's 128-position chunks in one fp32
    tensor-core accumulator before the split-K reduce, and the measured error grows linearly with that share: 1.1-1.4e-7
    per chunk on these operands (1 job at 48 x 48 with 9 chunks per CTA: 9.9e-7; 8 jobs at 96 x 96 with 262: 3.6e-5),
    while relative to A every element stays below 3.4e-7.  (The sums of random-sign data cancel: ||ref|| is ~1/sqrt(N)
    of ||A||, which is why rel-L2 is far larger than the error relative to A.)  The bound is 10x that slope."""
    lib = env[1]
    n_chunks = (B * (H + 1) * (W + 1) + 127) // 128
    grid = max(min(lib.sres_device_sm_count(), n_chunks * njobs), njobs)
    return WG_CHUNK * -(-n_chunks // (grid // njobs))


def check_job(tag, j, wb, bb=WG_B):
    """A job that owns all of its dw/db (cout_total 64, stride 1)."""
    ref, A = conv3x3_wgrad_ref(j.x, j.dy)
    refb, Ab = j.dy.double().sum((0, 2, 3)), j.dy.double().abs().sum((0, 2, 3))
    check_grad(f"{tag} dw", j.dw, ref * j.scale, A * j.scale, wb)
    if j.db is not None:
        check_grad(f"{tag} db", j.db, refb * j.scale, Ab * j.scale, bb)


GEOMS = [(64, 48, 48),      # x4 body and upsampler stage 0: 1201 chunks split unevenly over the jobs (148 CTAs: 19/18 for 8)
         (64, 96, 96),      # x4 upsampler stage 1: X window in 64-row boxes, 3-stage operand ring
         (2, 192, 192),     # x8 upsampler (96 x 96 tiles) at 192 x 192: 2-stage ring
         (1, 384, 384),     # x8 upsampler at 384 x 384: 1-stage ring
         (1, 5, 7)]         # a single 128-row chunk: grid = njobs


@pytest.mark.parametrize("njobs", [1, 3, 8])
@pytest.mark.parametrize("B,H,W", GEOMS)
def test_wgrad_batch_plain_jobs(env, B, H, W, njobs):
    """njobs independent 64 -> 64 gradients in one launch, each with its own x / dy, against fp64.  The 8-job batch runs
    twice and must be bit-identical (partials summed in a fixed order).
    Measured on a B200: rel-L2 dw 4e-8 (1 x 5 x 7) to 3.6e-5 (8 jobs at 64 x 96 x 96), see wg_bound; db <= 2.5e-7;
    max|err|/A <= 3.4e-7."""
    ws = workspace(env)
    jobs = plain_jobs(env, B, H, W, njobs)
    run_batch(env, jobs, B, H, W, ws)
    print(f"\n  wgrad batch {(B, H, W)} x {njobs} jobs")
    for i, j in enumerate(jobs):
        check_job(f"job {i}", j, wg_bound(env, B, H, W, njobs))
    if njobs == 8:
        first = [(j.dw.clone(), j.db.clone()) for j in jobs]
        for j in jobs:
            j.dw.fill_(float("nan"))
            j.db.fill_(float("nan"))
        run_batch(env, jobs, B, H, W, ws)
        for i, (j, (dw, db)) in enumerate(zip(jobs, first)):
            assert torch.equal(j.dw, dw) and torch.equal(j.db, db), f"job {i}: not bit-identical run to run"


def shuffle_jobs(env, B, H, W, f, subs, x, dw, db, seed=0):
    """The f*f sub-convolutions of a 64 -> f*f*64 upsampler conv, pushed like the backward pushes them: one shared x and
    dw/db, output channel n of sub-conv `sub` at oc = n*f*f + sub."""
    dev = env[2]
    g = _gen(dev, "shuffle", B, H, W, f, tuple(subs), seed)
    return [Job(x, _bf16(g, dev, B, 64, H, W), dw, db, cout_total=f * f * 64, stride=f * f, offset=s) for s in subs]


def shuffle_ref(jobs, f, cout):
    ref = torch.zeros(cout, 64, 3, 3, dtype=torch.float64, device=jobs[0].dw.device)
    A = torch.zeros_like(ref)
    refb = torch.zeros(cout, dtype=torch.float64, device=ref.device)
    Ab = torch.zeros_like(refb)
    for j in jobs:
        r, a = conv3x3_wgrad_ref(j.x, j.dy)
        ref[j.offset::f * f], A[j.offset::f * f] = r, a
        refb[j.offset::f * f] = j.dy.double().sum((0, 2, 3))
        Ab[j.offset::f * f] = j.dy.double().abs().sum((0, 2, 3))
    return ref, A, refb, Ab


def _x2_shuffle(env, B, H, W, tag):
    dev = env[2]
    ws = workspace(env)
    x = _bf16(_gen(dev, "x2x", B, H, W), dev, B, 64, H, W)
    dw = torch.full((256, 64, 3, 3), float("nan"), device=dev)
    db = torch.full((256,), float("nan"), device=dev)
    jobs = shuffle_jobs(env, B, H, W, 2, range(4), x, dw, db)
    run_batch(env, jobs, B, H, W, ws)
    ref, A, refb, Ab = shuffle_ref(jobs, 2, 256)
    print(f"\n  {tag} {(B, H, W)}: 4 sub-convs of a x2 PixelShuffle conv (cout 256, stride 4)")
    check_grad("dw (256,64,3,3)", dw, ref, A, wg_bound(env, B, H, W, 4))
    check_grad("db (256)", db, refb, Ab, WG_B)


@pytest.mark.parametrize("B,H,W", [(64, 48, 48), (64, 96, 96), (1, 5, 7)])
def test_wgrad_batch_pixelshuffle_x2(env, B, H, W):
    """The four sub-convolutions of a x2 upsampler conv (cout_total 256, oc_stride 4, oc_offset 0-3) in one batch sharing
    x and dw/db, as the backward issues them: every one of the 256 output channels against fp64.
    Measured on a B200: rel-L2 dw 4.3e-6 at 64 x 48 x 48, 1.8e-5 at 64 x 96 x 96 (see wg_bound), db <= 1.2e-7."""
    _x2_shuffle(env, B, H, W, "wgrad batch")


@pytest.mark.parametrize("B,H,W", [(64, 48, 48), (1, 5, 7)])
def test_wgrad_batch_pixelshuffle_x3(env, B, H, W):
    """The nine sub-convolutions of a x3 upsampler conv (cout_total 576, oc_stride 9) as an 8-job batch and a 1-job batch
    (how the backward's eight-job queue flushes them).  After the first batch the rows of sub-conv 8, which no job owns
    yet, still hold their NaN sentinel; after the second every row matches fp64.
    Measured on a B200: rel-L2 dw 8.9e-6 at 64 x 48 x 48 (see wg_bound), db <= 1.1e-7."""
    dev = env[2]
    ws = workspace(env)
    x = _bf16(_gen(dev, "x3x", B, H, W), dev, B, 64, H, W)
    dw = torch.full((576, 64, 3, 3), float("nan"), device=dev)
    db = torch.full((576,), float("nan"), device=dev)
    jobs = shuffle_jobs(env, B, H, W, 3, range(9), x, dw, db)
    run_batch(env, jobs[:8], B, H, W, ws)
    print(f"\n  wgrad batch {(B, H, W)}: 9 sub-convs of a x3 PixelShuffle conv (cout 576, stride 9) as 8 + 1 jobs")
    assert torch.isnan(dw[8::9]).all() and torch.isnan(db[8::9]).all(), "rows no job owns were written"
    own = torch.arange(576, device=dev) % 9 != 8
    ref, A, refb, Ab = shuffle_ref(jobs[:8], 3, 576)
    check_grad("dw rows of sub-convs 0-7", dw[own], ref[own], A[own], wg_bound(env, B, H, W, 8))
    check_grad("db rows of sub-convs 0-7", db[own], refb[own], Ab[own], WG_B)
    run_batch(env, jobs[8:], B, H, W, ws)
    ref, A, refb, Ab = shuffle_ref(jobs, 3, 576)
    check_grad("dw (576,64,3,3)", dw, ref, A, wg_bound(env, B, H, W, 8))
    check_grad("db (576)", db, refb, Ab, WG_B)


@pytest.mark.parametrize("B,H,W", [(64, 48, 48), (2, 192, 192), (1, 5, 7)])
def test_wgrad_batch_scale_accumulate_null_bias(env, B, H, W):
    """Per-job options in one batch: a plain job, scale = 0.1 (EDSR res_scale), accumulate = 1 into a prefilled dw/db,
    and dbias = NULL (that job's bias buffer is left untouched).
    Measured on a B200: rel-L2 dw <= 4.3e-6 (see wg_bound), db <= 1.3e-7."""
    dev = env[2]
    ws = workspace(env)
    jobs = plain_jobs(env, B, H, W, 4, seed=1)
    jobs[1].scale = SCALE
    jobs[2].acc = 1
    pre_w = torch.randn(64, 64, 3, 3, device=dev) * 100
    pre_b = torch.randn(64, device=dev) * 100
    jobs[2].dw.copy_(pre_w)
    jobs[2].db.copy_(pre_b)
    untouched = jobs[3].db
    jobs[3].db = None
    jobs[3].scale = SCALE
    run_batch(env, jobs, B, H, W, ws)
    print(f"\n  wgrad batch {(B, H, W)}: plain | scale 0.1 | accumulate | dbias NULL + scale 0.1")
    wb = wg_bound(env, B, H, W, 4)
    check_job("plain dw/db", jobs[0], wb)
    check_job("scale 0.1", jobs[1], wb)
    ref, A = conv3x3_wgrad_ref(jobs[2].x, jobs[2].dy)
    check_grad("accumulate dw", jobs[2].dw, pre_w.double() + ref, A + pre_w.double().abs(), wb)
    check_grad("accumulate db", jobs[2].db, pre_b.double() + jobs[2].dy.double().sum((0, 2, 3)),
               jobs[2].dy.double().abs().sum((0, 2, 3)) + pre_b.double().abs(), WG_B)
    check_job("dbias NULL", jobs[3], wb)
    assert torch.isnan(untouched).all()


def test_wgrad_batches_back_to_back(env):
    """Three batches enqueued on one workspace and stream with no host synchronisation between them, as the backward
    issues them (the next batch's CTAs overwrite the split-K partials behind programmatic dependent launch while the
    previous reduce may still read them): a 4-job batch at 96 x 96, then an 8-job and a 3-job batch at 48 x 48.  Each
    result is bit-identical to the same batch run alone, and matches fp64."""
    ws = workspace(env)
    batches = [((64, 96, 96), plain_jobs(env, 64, 96, 96, 4, seed=2)), ((64, 48, 48), plain_jobs(env, 64, 48, 48, 8, seed=2)),
               ((64, 48, 48), plain_jobs(env, 64, 48, 48, 3, seed=3))]
    alone = []
    for geom, jobs in batches:
        run_batch(env, jobs, *geom, ws)
        alone.append([(j.dw.clone(), j.db.clone()) for j in jobs])
        for j in jobs:
            j.dw.fill_(float("nan"))
            j.db.fill_(float("nan"))
    for geom, jobs in batches:
        run_batch(env, jobs, *geom, ws, sync=False)
    torch.cuda.synchronize()
    print("\n  wgrad batches back to back on one workspace")
    for k, ((geom, jobs), ref) in enumerate(zip(batches, alone)):
        for i, (j, (dw, db)) in enumerate(zip(jobs, ref)):
            assert torch.equal(j.dw, dw) and torch.equal(j.db, db), f"batch {k} job {i} differs from the batch run alone"
            check_job(f"batch {k} {geom} job {i}", j, wg_bound(env, *geom, len(jobs)))


def test_wgrad_batch_n128_tap_table(env, monkeypatch):
    """The opt-in four-taps-per-MMA scheme (SRES_WGRAD_N128=1, read per call) scatters through its own tap table: 8 plain
    jobs and the x2 PixelShuffle batch at 48 x 48 against fp64 (same bounds as the default scheme).
    Measured on a B200: x2 PixelShuffle rel-L2 dw 4.3e-6, db 1.2e-7."""
    monkeypatch.setenv("SRES_WGRAD_N128", "1")
    B, H, W = 64, 48, 48
    ws = workspace(env)
    jobs = plain_jobs(env, B, H, W, 8, seed=4)
    run_batch(env, jobs, B, H, W, ws)
    print(f"\n  wgrad batch {(B, H, W)} x 8 jobs, SRES_WGRAD_N128=1")
    for i, j in enumerate(jobs):
        check_job(f"job {i}", j, wg_bound(env, B, H, W, 8))
    _x2_shuffle(env, B, H, W, "SRES_WGRAD_N128=1")


# ---------------------------------------------------------------------------------------------------------------------
# B. head and tail weight gradients (CUDA cores, fp32)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,Cs,H,W", [(64, 2, 192, 192),    # x4 tail at B = 64
                                      (1, 4, 768, 768),     # x8 tail: three column strips, the warps split 4 channels
                                      (2, 1, 40, 514),      # three strips, W % 4 != 0: scalar path
                                      (2, 3, 48, 300),      # Cs = 3, two strips, vector path
                                      (3, 3, 20, 22)])      # Cs = 3, one strip, scalar path
def test_small_out_wgrad(env, B, Cs, H, W):
    """Tail conv (64 -> Cs) weight/bias gradient from the planar fp32 output gradient and the bf16 PTL conv input, against
    fp64; then accumulate = 1 with db = NULL: dw doubles and db keeps its value bit for bit.
    Measured on a B200: rel-L2 dw <= 6.0e-7, db <= 4.8e-7; max|err|/A <= 2e-8."""
    L, lib, dev = env
    g = _gen(dev, "small_out", B, Cs, H, W)
    u = _bf16(g, dev, B, 64, H, W)
    dout = torch.randn(B, Cs, H, W, device=dev, generator=g)
    up = to_ptl(u, torch.bfloat16)
    wsb = lib.sres_small_wgrad_workspace_bytes()
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    dw = torch.full((Cs, 64, 3, 3), float("nan"), device=dev)
    db = torch.full((Cs,), float("nan"), device=dev)
    L.check(lib.sres_small_out_wgrad(ptr(dout), ptr(up), B, Cs, H, W, ptr(dw), ptr(db), 0, ptr(ws), C.c_size_t(wsb),
                                     L.cur_stream()), "small_out_wgrad")
    torch.cuda.synchronize()
    ref, A = conv3x3_wgrad_ref(u, dout)
    print(f"\n  small_out_wgrad {(B, Cs, H, W)}")
    check_grad("dw", dw, ref, A, SO_W)
    check_grad("db", db, dout.double().sum((0, 2, 3)), dout.double().abs().sum((0, 2, 3)), SO_B)
    db1 = db.clone()
    L.check(lib.sres_small_out_wgrad(ptr(dout), ptr(up), B, Cs, H, W, ptr(dw), None, 1, ptr(ws), C.c_size_t(wsb),
                                     L.cur_stream()), "small_out_wgrad")
    torch.cuda.synchronize()
    check_grad("dw, accumulate = 1", dw, 2 * ref, 2 * A, SO_W)
    assert torch.equal(db, db1), "db = NULL must leave the bias gradient alone"


@pytest.mark.parametrize("B,Cs,H,W", [(64, 2, 48, 48),      # x4 head at B = 64: band kernel
                                      (2, 4, 96, 96),       # band kernel, 4 channels
                                      (2, 3, 50, 51)])      # W % 4 != 0: scalar kernel, 5304 positions wrap its 2368-wide grid stride
def test_small_in_wgrad(env, B, Cs, H, W):
    """Head conv (Cs -> 64) weight/bias gradient from two fp32 PTL gradient addends and the planar input, against fp64;
    then g2 = NULL, accumulate = 1, db = NULL: dw grows by the g1 gradient and db keeps its value bit for bit.
    Measured on a B200: rel-L2 dw <= 4.7e-7, db <= 4.4e-7; max|err|/A <= 6.3e-8."""
    L, lib, dev = env
    g = _gen(dev, "small_in", B, Cs, H, W)
    x = torch.randn(B, Cs, H, W, device=dev, generator=g)
    g1 = torch.randn(B, 64, H, W, device=dev, generator=g)
    g2 = torch.randn(B, 64, H, W, device=dev, generator=g)
    g1p, g2p = to_ptl(g1, torch.float32), to_ptl(g2, torch.float32)
    wsb = lib.sres_small_wgrad_workspace_bytes()
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    dw = torch.full((64, Cs, 3, 3), float("nan"), device=dev)
    db = torch.full((64,), float("nan"), device=dev)
    L.check(lib.sres_small_in_wgrad(ptr(g1p), ptr(g2p), ptr(x), B, Cs, H, W, ptr(dw), ptr(db), 0, ptr(ws), C.c_size_t(wsb),
                                    L.cur_stream()), "small_in_wgrad")
    torch.cuda.synchronize()
    gs = g1.double() + g2.double()
    ref, A = conv3x3_wgrad_ref(x, gs)
    print(f"\n  small_in_wgrad {(B, Cs, H, W)}")
    check_grad("dw (g1 + g2)", dw, ref, A, SI_W)
    check_grad("db (g1 + g2)", db, gs.sum((0, 2, 3)), gs.abs().sum((0, 2, 3)), SI_B)
    dw1, db1 = dw.clone(), db.clone()
    L.check(lib.sres_small_in_wgrad(ptr(g1p), None, ptr(x), B, Cs, H, W, ptr(dw), None, 1, ptr(ws), C.c_size_t(wsb),
                                    L.cur_stream()), "small_in_wgrad")
    torch.cuda.synchronize()
    ref1, A1 = conv3x3_wgrad_ref(x, g1)
    check_grad("dw += (g1 only)", dw, dw1.double() + ref1, A1 + dw1.double().abs(), SI_W)
    assert torch.equal(db, db1), "db = NULL must leave the bias gradient alone"


# ---------------------------------------------------------------------------------------------------------------------
# C. channel attention
# ---------------------------------------------------------------------------------------------------------------------
def ca_forward64(m, w1, b1, w2, b2):
    """s = sigmoid(W2 relu(W1 m + b1) + b2) in float64, batched: m (..., B, 64), w1 (..., hid, 64), w2 (..., 64, hid)."""
    h = torch.relu(m @ w1.transpose(-1, -2) + b1.unsqueeze(-2))
    return torch.sigmoid(h @ w2.transpose(-1, -2) + b2.unsqueeze(-2)), h


@pytest.mark.parametrize("B", [1, 33, 64])
@pytest.mark.parametrize("hid", [4, 32, 64])
def test_ca_param_grads_twenty_layers(env, hid, B):
    """Squeeze-excite parameter gradients of a residual group's 20 CALayers in one call, at the real RCAB parameter stride
    2(64*64*9 + 64) + 2*64*hid + hid + 64 (B = 33 and 64 take two 32-image shared-memory chunks), against fp64 autograd
    of sigmoid(W2 relu(W1 m + b1) + b2) with upstream ds.  First accumulate = 1 onto prefilled slices, then
    accumulate = 0; the conv-weight slots between the slices keep their sentinel bit for bit.
    Measured on a B200 (worst layer of any case): rel-L2 <= 6.3e-7 for B > 1, 4.5e-6 at B = 1 (see CA_P_B1); every
    element within 1.2e-6 A.  This test found sigmoid'(z) computed as
    s * (1 - s): 1 - s cancels where s nears 1, and at B = 1 single elements of dw2 / db2 were off by 4.8e-4 A."""
    L, lib, dev = env
    R = 20
    stride = 2 * (KW + 64) + 2 * 64 * hid + hid + 64
    off = 2 * (KW + 64)
    n_ca = 2 * 64 * hid + hid + 64
    g = _gen(dev, "ca_param", hid, B)
    params = torch.randn(R, stride, device=dev, generator=g) * 0.3
    mean = torch.randn(R, B, 64, device=dev, generator=g)
    ds = torch.randn(R, B, 64, device=dev, generator=g)
    SENT = 1234.5
    grads = torch.full((R, stride), SENT, device=dev)
    prefill = torch.randn(R, n_ca, device=dev, generator=g) * 10
    grads[:, off:] = prefill
    scr = torch.empty(lib.sres_ca_param_grads_scratch_bytes(R, B), dtype=torch.uint8, device=dev)

    # fp64 reference, all layers at once: autograd for the values; for the conditioning A the same chain over absolute
    # values (|dz| through |W2| gives the scale of dh, |W1||m| + |b1| that of h)
    ca = params[:, off:].double()
    w1 = ca[:, :hid * 64].reshape(R, hid, 64).clone().requires_grad_(True)
    b1 = ca[:, hid * 64:hid * 65].clone().requires_grad_(True)
    w2 = ca[:, hid * 65:hid * 129].reshape(R, 64, hid).clone().requires_grad_(True)
    b2 = ca[:, hid * 129:].clone().requires_grad_(True)
    m = mean.double()
    s, h = ca_forward64(m, w1, b1, w2, b2)
    (ds.double() * s).sum().backward()
    ref = torch.cat([w1.grad.reshape(R, -1), b1.grad, w2.grad.reshape(R, -1), b2.grad], 1)
    with torch.no_grad():
        dzA = (ds.double() * s * (1 - s)).abs()
        dhA = (dzA @ w2.abs()) * (h > 0)
        hA = (m.abs() @ w1.abs().transpose(1, 2) + b1.abs().unsqueeze(1)) * (h > 0)
        A = torch.cat([(dhA.transpose(1, 2) @ m.abs()).reshape(R, -1), dhA.sum(1), (dzA.transpose(1, 2) @ hA).reshape(R, -1),
                       dzA.sum(1)], 1)
    pieces = [("w1", 0, hid * 64), ("b1", hid * 64, hid * 65), ("w2", hid * 65, hid * 129), ("b2", hid * 129, n_ca)]

    bound = CA_P_B1 if B == 1 else CA_P
    print(f"\n  ca_param_grads hid {hid} B {B}, 20 layers")
    for acc in (1, 0):
        L.check(lib.sres_ca_param_grads(ptr(params[0, off:]), ptr(grads[0, off:]), C.c_int64(stride), R, ptr(mean), ptr(ds), B,
                                        hid, acc, ptr(scr), C.c_size_t(scr.numel()), L.cur_stream()), "ca_param_grads")
        torch.cuda.synchronize()
        assert bool((grads[:, :off] == SENT).all()), "conv-weight slots between the CA slices were written"
        base = prefill.double() if acc else torch.zeros_like(ref)
        for name, a, b in pieces:
            got, exp, cond = grads[:, off + a:off + b], base[:, a:b] + ref[:, a:b], A[:, a:b] + base[:, a:b].abs()
            rel = ((got.double() - exp).norm(dim=1) / exp.norm(dim=1)).nan_to_num(0.0)
            worst = int(rel.argmax())
            check_grad(f"accumulate {acc}: {name} (layer {worst}, the worst of 20)", got[worst], exp[worst], cond[worst], bound)
            assert bool((rel < bound).all()) and bool(((got.double() - exp).abs() <= 2.0 ** -12 * cond).all()), name


@pytest.mark.parametrize("B,H,W,hid", [(64, 48, 48, 4),     # x4 training tiles, RCAN-full reduction 16
                                       (3, 20, 24, 32),
                                       (5, 10, 11, 64)])    # (H+1)(W+1) = 132: almost every M tile straddles two images
def test_ca_bwd_apply(env, B, H, W, hid):
    """The CALayer backward the training step takes for (H+1)(W+1) >= 128, where ds = sum(g * t2) arrives as per-tile
    partial sums of the convolution that produced g.  tile_part is built here from fp64 products g * t2, row by row, in
    the layout [tile][segment][quarter][64] with tile_rows = sres_conv_tile_rows(H, W), the rows spread unevenly over
    the four quarters; (tile, segment) slots that hold no rows are NaN.  save_ds must match the fp64 sum, dt2 must be
    within one bf16 rounding of fp64 g*s + dm/(HW) and zero on every padding row.
    Measured on a B200: rel-L2 save_ds <= 9.7e-8, max|err|/A <= 3.4e-8."""
    L, lib, dev = env
    RP = (H + 1) * (W + 1)
    rows = B * RP
    TR = lib.sres_conv_tile_rows(H, W)
    nt = lib.sres_conv_mtiles(B, H, W)
    assert nt == (rows + TR - 1) // TR
    g = _gen(dev, "ca_bwd_apply", B, H, W, hid)
    t2 = _bf16(g, dev, B, 64, H, W)
    t2p = to_ptl(t2, torch.bfloat16)
    grad = torch.randn(rows, 64, device=dev, generator=g)        # padding rows too: dt2 must still be 0 there
    w1, b1 = torch.randn(hid, 64, device=dev, generator=g) * 0.3, torch.randn(hid, device=dev, generator=g)
    w2, b2 = torch.randn(64, hid, device=dev, generator=g) * 0.3, torch.randn(64, device=dev, generator=g)
    mean = torch.randn(B, 64, device=dev, generator=g) * 0.5

    prod = grad.double() * t2p.double()
    q = torch.arange(rows, device=dev)
    t = q // TR
    seg = q // RP - (t * TR) // RP
    assert int(seg.max()) <= 1
    quarter = torch.multinomial(torch.tensor([0.55, 0.25, 0.15, 0.05], device=dev), rows, replacement=True, generator=g)
    slot = (t * 2 + seg) * 4 + quarter
    part = torch.zeros(nt * 8, 64, dtype=torch.float64, device=dev).index_add_(0, slot, prod)
    used = torch.zeros(nt * 2, dtype=torch.float64, device=dev).index_add_(0, t * 2 + seg, torch.ones(rows, dtype=torch.float64, device=dev))
    part = part.reshape(nt, 2, 4, 64)
    part[(used == 0).reshape(nt, 2)] = float("nan")
    tile_part = part.float().contiguous()

    dt2 = torch.full((rows, 64), 7.0, device=dev, dtype=torch.bfloat16)
    save_ds = torch.full((B, 64), float("nan"), device=dev)
    L.check(lib.sres_ca_bwd_apply(ptr(grad), ptr(tile_part), ptr(w1), ptr(b1), ptr(w2), ptr(b2), hid, ptr(mean), ptr(dt2),
                                  ptr(save_ds), B, H, W, L.cur_stream()), "ca_bwd_apply")
    torch.cuda.synchronize()

    ds_ref = prod.reshape(B, RP, 64).sum(1)
    A_ds = (grad.double() * t2p.double()).abs().reshape(B, RP, 64).sum(1)
    print(f"\n  ca_bwd_apply {(B, H, W)} hid {hid}, tile_rows {TR}, {nt} tiles")
    check_grad("save_ds", save_ds, ds_ref, A_ds, CA_DS)

    m = mean.double().requires_grad_(True)
    s, h = ca_forward64(m, w1.double(), b1.double(), w2.double(), b2.double())
    (ds_ref * s).sum().backward()
    with torch.no_grad():
        gs = grad.double().reshape(B, RP, 64) * s.unsqueeze(1)
        dm = (m.grad / (H * W)).unsqueeze(1)
        ref = (gs + dm).reshape(rows, 64)
        # one bf16 rounding (half an ulp <= 2^-8 |v|) plus room for the fp32 arithmetic before it, judged against the
        # scale of each term (dm through the chain over absolute values, from A of ds)
        dmA = (((A_ds * s * (1 - s)) @ w2.double().abs()) * (h > 0)) @ w1.double().abs() / (H * W)
        slack = 2.0 ** -8 * ref.abs() + 2.0 ** -16 * (gs.abs() + dmA.unsqueeze(1)).reshape(rows, 64)
    valid = torch.zeros(B, H + 1, W + 1, dtype=torch.bool, device=dev)
    valid[:, :H, :W] = True
    valid = valid.reshape(rows)
    err = (dt2.double() - ref).abs()[valid]
    print(f"  {'dt2 (valid rows)':<44s} max|err|/|ref| {(err / ref.abs()[valid]).max().item():.2e} (one bf16 rounding: 2^-8 = 3.9e-03)")
    assert bool((err <= slack[valid]).all()), "dt2 is more than one bf16 rounding away from fp64 g*s + dm/(HW)"
    assert pads_are_zero(dt2, B, H, W)
