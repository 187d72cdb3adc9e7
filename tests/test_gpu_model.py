"""GPU parity of the whole path: model forward/backward/Adam vs the oracle and the reference's golden
vectors, tile extraction / normalisation / flip / stitching bit-exact vs the oracle, and the mirror of
the reference controller API end to end.  Floating-point tolerance (BASELINE.json north_star): global
rel-L2 <= 1e-2 on outputs and on the full gradient (bf16 operands, fp32 accumulation)."""
import os
import random

import numpy as np
import pytest
import torch

import rcan_oracle as O
import tiles_oracle as T
from gpu_util import rel_l2
from synth import MODEL_CASES, TILE_CASES, golden_file, sha, synth_hr, synth_region

pytestmark = pytest.mark.gpu
TOL = 1e-2


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda:0")


def _build(cfg, C, dev_):
    from sres_b200 import nn as snn
    if O.is_edsr(cfg):
        return snn.EDSR(nchannels_in=C, nchannels_out=C, nfeatures=64, nlayers=cfg["nlayers"], scale=O.scale_of(cfg),
                        res_scale=cfg["res_scale"], device=dev_)
    return snn.RCAN(nchannels_in=C, nchannels_out=C, nfeatures=64, nlayers=cfg["nlayers"], nblocks=cfg["nblocks"],
                    cbottleneck=cfg["cbottleneck"], scale=O.scale_of(cfg), device=dev_)


@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_train_step_matches_oracle_and_golden(name, dev, golden_dir):
    from sres_b200 import nn as snn
    over, B, S, C, loss_name, smooth, full_out = MODEL_CASES[name]
    gold = np.load(os.path.join(golden_dir, golden_file(name)))
    cfg = O.model_cfg(**over)
    scale = O.scale_of(cfg)
    sd = O.make_state_dict(cfg, C, C)
    hr = synth_hr(B, C, S * scale, smooth=smooth)
    loss_o, prd_o, grads_o = O.loss_and_grads(hr, sd, cfg, loss_name)
    model = _build(cfg, C, dev)
    assert [k for k, _ in model.named_parameters()] == list(sd.keys()) == [str(n) for n in gold["grad_names"]]
    model.load_state_dict(sd)
    opt = snn.FusedAdam(model, lr=1e-4)
    hr_d = hr.to(dev)
    lr_d = snn.bicubic_resize(hr_d, 1.0 / scale)
    assert (lr_d.cpu()[: gold["lr_input"].shape[0]] - torch.from_numpy(gold["lr_input"])).abs().max() < 2e-6
    prd = model(lr_d.requires_grad_(True))
    loss = snn.loss(prd, hr_d, loss_name)
    loss.backward()
    # vs oracle
    assert rel_l2(prd.detach().cpu(), prd_o) < TOL
    assert abs(loss.item() - loss_o) < TOL * abs(loss_o)
    num = sum((p.grad.cpu() - grads_o[k]).double().pow(2).sum().item() for k, p in model.named_parameters())
    den = sum(g.double().pow(2).sum().item() for g in grads_o.values())
    assert (num / den) ** 0.5 < TOL
    # vs the reference's own numbers (golden fixture)
    out = prd.detach().cpu().numpy() if full_out else prd.detach().cpu().numpy()[:, :, ::8, ::8]
    assert np.linalg.norm(out - gold["output"]) / np.linalg.norm(gold["output"]) < TOL
    assert abs(loss.item() - float(gold["loss"])) < TOL * float(gold["loss"])
    gn = np.array([p.grad.double().norm().item() for _, p in model.named_parameters()])
    big = gold["grad_norms"] > 0.05 * gold["grad_norms"].max()
    np.testing.assert_allclose(gn[big], gold["grad_norms"][big], rtol=3e-2)
    # every tensor the fixture holds in full -- conv and channel-attention weights and biases at both ends of the body, head and
    # tail: per-tensor rel-L2 against the REFERENCE's gradient, <= 2e-2 each (measured 4e-4 ... 1.2e-2).  One documented
    # exception (DESIGN.md section 4, deviation 3): the bias of an RCAB's FIRST conv in the white-noise cases on 8..12-pixel
    # tiles.  Its gradient is sum_q relu'(t1[q]) * g[q] over only ~150-300 positions with random signs; bf16 operand rounding
    # flips the ReLU mask of about one position in 300 and ONE flipped term moves such a cancellation-heavy sum by a few %
    # (measured 3.9e-2 ... 5.3e-2).  With smooth fields / 48-pixel tiles (2304+ positions) the same tensors sit at 3e-3 ... 8e-3.
    params = dict(model.named_parameters())
    worst = {}
    for gk in [k for k in gold.files if k.startswith("grad::") and "[" not in k]:
        key = gk[len("grad::"):]
        g = params[key].grad.cpu().numpy()
        worst[key] = float(np.linalg.norm(g - gold[gk]) / (np.linalg.norm(gold[gk]) + 1e-30))
    print(name, "per-tensor gradient rel-L2 vs reference:", {k: f"{v:.2e}" for k, v in worst.items()})
    for key, err in worst.items():
        conv1_bias = key.endswith(".body.0.bias") and not smooth
        assert err < (8 * TOL if conv1_bias else 2 * TOL), (key, err, worst)
    # one fused Adam step from the GPU's OWN gradients against the reference's post-step parameters.  The first Adam step
    # moves every element by lr * g / (|g| + eps), i.e. by +-lr wherever |g| >> eps: the update direction only differs where
    # a gradient element is within rounding distance of zero.
    pre = {k: p.detach().clone() for k, p in model.named_parameters()}
    opt.step()
    torch.cuda.synchronize()
    frac_off = {}
    for pk in [k for k in gold.files if k.startswith("post::")]:
        key = pk[len("post::"):]
        d_gpu = (params[key].detach() - pre[key]).cpu().numpy()
        d_ref = gold[pk] - sd[key].numpy()
        assert np.abs(d_gpu).max() <= 1.0001e-4 and np.abs(d_ref).max() <= 1.0001e-4
        n_off = int((np.abs(d_gpu - d_ref) > 2e-5).sum())
        frac_off[key] = n_off / d_ref.size
        assert n_off <= max(2, d_ref.size // 100), (key, n_off, d_ref.size)     # measured: 0-2 elements, <= 0.9 % of big tensors
    print(name, "fraction of elements whose first Adam update differs from the reference's:", {k: f"{v:.1e}" for k, v in frac_off.items()})
    gpost = np.array([p.detach().double().norm().item() for _, p in model.named_parameters()])
    np.testing.assert_allclose(gpost, gold["post_norms"], rtol=5e-4)   # every parameter tensor after the GPU-computed step
    # one fused Adam step from the oracle's gradients must reproduce the oracle's Adam
    model.load_state_dict(O.make_state_dict(cfg, C, C))
    opt = snn.FusedAdam(model, lr=1e-4)
    with torch.no_grad():
        for k, p in model.named_parameters():
            p.grad.copy_(grads_o[k])
    opt.step()
    adam = O.AdamState(sd, lr=1e-4)
    with torch.no_grad():
        adam.step(sd, grads_o)
    for k, p in model.named_parameters():
        assert (p.detach().cpu() - sd[k]).abs().max() < 1e-6, k
    # inference mode (no grad) runs the same kernels without saved activations
    model.load_state_dict(O.make_state_dict(cfg, C, C))
    with torch.no_grad():
        prd2 = model(lr_d.detach())
    assert rel_l2(prd2.cpu(), prd_o) < TOL


@pytest.mark.parametrize("nblocks", [1, 20])
def test_x8_wide_tiles_forward_and_backward_run(dev, nblocks):
    """BASELINE config 5 geometry (x8, 4 channels, 96x96 LR -> 768x768 HR) at batch 1, with one RCAB and with one FULL
    residual group (20 RCABs + group conv, reduction 16): three PixelShuffle stages up to 768-pixel rows, where the tail
    conv runs on the narrow three-taps-per-MMA kernel.  Output, loss and the full gradient against the oracle."""
    from sres_b200 import nn as snn
    cfg = O.model_cfg(nlayers=1, nblocks=nblocks, cbottleneck=16 if nblocks > 1 else 2, downscale_factors=[2, 2, 2])
    sd = O.make_state_dict(cfg, 4, 4)
    hr = synth_hr(1, 4, 768, smooth=True)
    loss_o, prd_o, grads_o = O.loss_and_grads(hr, sd, cfg, "l2")
    model = _build(cfg, 4, dev)
    model.load_state_dict(sd)
    hr_d = hr.to(dev)
    prd = model(snn.bicubic_resize(hr_d, 1.0 / 8).requires_grad_(True))
    loss = snn.loss(prd, hr_d, "l2")
    loss.backward()
    assert prd.shape == (1, 4, 768, 768) and rel_l2(prd.detach().cpu(), prd_o) < TOL
    num = sum((p.grad.cpu() - grads_o[k]).double().pow(2).sum().item() for k, p in model.named_parameters())
    den = sum(g.double().pow(2).sum().item() for g in grads_o.values())
    assert (num / den) ** 0.5 < TOL and abs(loss.item() - loss_o) < TOL * abs(loss_o)


def test_full_depth_parity_vs_oracle(dev):
    """RCAN-full depth (10 groups x 20 RCABs, reduction 16, x4) against the CPU oracle on a batch the oracle finishes in
    seconds: outputs, loss and the global gradient within the 1e-2 parity tolerance (SURVEY 8d expects ~7e-3)."""
    from sres_b200 import nn as snn
    cfg = O.model_cfg(cbottleneck=16)
    sd = O.make_state_dict(cfg, 2, 2)
    hr = synth_hr(2, 2, 192, smooth=True)
    loss_o, prd_o, grads_o = O.loss_and_grads(hr, sd, cfg, "l2")
    model = _build(cfg, 2, dev)
    model.load_state_dict(sd)
    hr_d = hr.to(dev)
    prd = model(snn.bicubic_resize(hr_d, 0.25).requires_grad_(True))
    loss = snn.loss(prd, hr_d, "l2")
    loss.backward()
    num = sum((p.grad.cpu() - grads_o[k]).double().pow(2).sum().item() for k, p in model.named_parameters())
    den = sum(g.double().pow(2).sum().item() for g in grads_o.values())
    ro, rg = rel_l2(prd.detach().cpu(), prd_o), (num / den) ** 0.5
    print(f"full depth: output rel-L2 {ro:.3e}, gradient rel-L2 {rg:.3e}, loss {loss.item():.6f} vs {loss_o:.6f}")
    assert ro < TOL and rg < TOL and abs(loss.item() - loss_o) < TOL * abs(loss_o)


def test_full_size_properties(dev):
    """BASELINE config 2 at full size (RCAN-full x4, 64 tiles of 2x48x48): too big for the CPU oracle in a test, so the
    size-independent properties the path offers are checked instead -- tiles are independent units (a batch equals its
    halves), backward is linear in the output gradient and additive over tiles, the tail-bias gradient is the plain sum
    of the output gradient, and everything is bit-reproducible run to run (fixed-order reductions, no atomics)."""
    from sres_b200 import nn as snn
    torch.manual_seed(5)
    model = snn.RCAN(nchannels_in=2, nchannels_out=2, nfeatures=64, nlayers=10, nblocks=20, cbottleneck=16, scale=4, device=dev)
    eng = model.engine
    x = torch.randn(64, 2, 48, 48, device=dev)
    dout = torch.randn(64, 2, 192, 192, device=dev) * 1e-3

    def run(xb, db):
        out = eng.forward(xb, training=True).clone()
        eng.backward(xb, db, accumulate=False)
        return out, eng.flat_grad.clone()

    out, g = run(x, dout)
    out2, g2 = run(x, dout)
    assert torch.isfinite(out).all() and torch.isfinite(g).all()
    assert torch.equal(out, out2) and torch.equal(g, g2), "forward / backward must be bit-reproducible"
    oa, ga = run(x[:32].contiguous(), dout[:32].contiguous())
    ob, gb = run(x[32:].contiguous(), dout[32:].contiguous())
    # Not bit-equal: the pooled means are summed per 128-row tile and tile boundaries fall differently in a different
    # batch; a last-bit difference there flips bf16 roundings downstream and 200 RCABs amplify it to the same few 1e-3
    # that separate the bf16 path from the fp32 oracle.  The bound is the parity tolerance.
    ra, rb = rel_l2(torch.cat([oa, ob]), out), rel_l2(ga + gb, g)
    _, g3 = run(x, 3.0 * dout)
    rc = rel_l2(g3, 3.0 * g)              # linear up to the bf16 rounding of the gradient operands
    print(f"full size: batch-split outputs {ra:.3e}, gradient additivity {rb:.3e}, linearity {rc:.3e}")
    # (white-noise weights, inputs and output gradient are the worst case for this sensitivity: 3x the parity tolerance)
    assert ra < TOL and rb < 3 * TOL and rc < 3 * TOL
    names = [k for k, _ in eng.layout]
    off = sum(int(np.prod(s_)) for _, s_ in eng.layout[:names.index("tail.1.bias")])
    assert rel_l2(g[off:off + 2], dout.sum((0, 2, 3))) < 1e-5


def test_full_size_batch_tiles_match_oracle(dev):
    """BASELINE config 2 at full size (RCAN-full x4, reduction 16, 64 tiles of 2x48x48) against the ORACLE: tiles are
    independent units, so the oracle runs on four of the 64 tiles and must reproduce those four outputs of the batch-64 GPU
    pass; with an output gradient that is zero outside those tiles the batch-64 parameter gradients equal the oracle's
    gradients of the four-tile problem (head, tail, channel-attention and conv tensors compared one by one, the
    full gradient globally)."""
    cfg = O.model_cfg(cbottleneck=16)
    sd = O.make_state_dict(cfg, 2, 2)
    model = _build(cfg, 2, dev)
    model.load_state_dict(sd)
    eng = model.engine
    from sres_b200 import nn as snn
    hr = synth_hr(64, 2, 192, smooth=True)
    x = snn.bicubic_resize(hr.to(dev), 0.25).contiguous()
    pick = [0, 21, 42, 63]
    out = eng.forward(x, training=True).clone()
    # oracle on the four tiles (fp32 CPU restatement of the reference network + autograd); the output gradient is the
    # RMSE gradient of the four-tile problem (stats.py:5-8), handed to both sides
    xs = x[pick].cpu()
    prd4 = O.model_forward(xs, sd, cfg)
    diff = prd4 - hr[pick]
    dsel = (diff / (diff.numel() * torch.sqrt((diff * diff).mean()))).contiguous()
    prd_o, grads_o = O.forward_backward(xs, dsel, sd, cfg)
    dout = torch.zeros(64, 2, 192, 192)
    dout[pick] = dsel
    eng.backward(x, dout.to(dev), accumulate=False)
    grad = eng.flat_grad.clone().cpu()
    assert rel_l2(out[pick].cpu(), prd_o) < TOL
    off, num, den, per = 0, 0.0, 0.0, {}
    for k, shp in eng.layout:
        n = int(np.prod(shp))
        gg, go = grad[off:off + n].double(), grads_o[k].reshape(-1).double()
        num += (gg - go).pow(2).sum().item(); den += go.pow(2).sum().item()
        if k in ("head.0.weight", "head.0.bias", "tail.1.weight", "tail.1.bias", "tail.0.0.weight", "body.10.weight",
                 "body.0.body.0.body.3.conv_du.0.weight", "body.9.body.19.body.3.conv_du.2.bias", "body.9.body.20.bias",
                 "body.4.body.7.body.2.weight"):
            per[k] = float((gg - go).norm() / (go.norm() + 1e-30))
        off += n
    print(f"batch 64, four tiles vs oracle: output {rel_l2(out[pick].cpu(), prd_o):.3e}, gradient {(num / den) ** 0.5:.3e},",
          {k: f"{v:.2e}" for k, v in per.items()})
    assert (num / den) ** 0.5 < TOL and max(per.values()) < 2 * TOL, per


def test_gradient_accumulation_and_stock_adam(dev):
    """Two backward passes without zero_grad accumulate (autograd semantics); torch.optim.Adam works on the
    parameter views and its in-place update is picked up by the next forward (weights are re-packed)."""
    from sres_b200 import nn as snn
    cfg = O.model_cfg(nlayers=1, nblocks=1)
    model = _build(cfg, 2, dev)
    model.load_state_dict(O.make_state_dict(cfg, 2, 2))
    x = torch.randn(2, 2, 12, 12, device=dev)
    tgt = torch.randn(2, 2, 48, 48, device=dev)
    snn.loss(model(x.requires_grad_(True)), tgt, "l2").backward()
    g1 = model.engine.flat_grad.clone()
    snn.loss(model(x), tgt, "l2").backward()
    assert rel_l2(model.engine.flat_grad, 2 * g1) < 1e-5
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    out0 = model(x).detach().clone()
    opt.step()
    out1 = model(x).detach()
    assert (out1 - out0).abs().max() > 1e-4
    opt.zero_grad()
    assert all(p.grad is None for p in model.parameters())
    snn.loss(model(x), tgt, "l2").backward()
    assert all(p.grad is not None for p in model.parameters())


def test_fused_adam_state_interchanges_with_torch_adam(dev, tmp_path):
    """FusedAdam.state_dict() has torch.optim.Adam's layout (what the reference's CheckpointManager saves,
    checkpoints.py:20,44): a stock Adam loads it and continues exactly like FusedAdam does, and the other way round;
    a state that does not fit raises before anything is modified."""
    from sres_b200 import nn as snn
    cfg = O.model_cfg(nlayers=1, nblocks=2)
    sd0 = O.make_state_dict(cfg, 2, 2)
    x = torch.randn(2, 2, 12, 12, device=dev)
    tgt = torch.randn(2, 2, 48, 48, device=dev)

    def run(model, opt, nsteps):
        for _ in range(nsteps):
            opt.zero_grad()
            snn.loss(model(x.clone().requires_grad_(True)), tgt, "l2").backward()
            opt.step()

    a = _build(cfg, 2, dev); a.load_state_dict(sd0)
    oa = snn.FusedAdam(a, lr=1e-3, weight_decay=1e-4)
    run(a, oa, 3)
    state = oa.state_dict()
    ref_layout = torch.optim.Adam(a.parameters(), lr=1e-3).state_dict()
    assert set(state) == {"state", "param_groups"} and set(state["param_groups"][0]) == set(ref_layout["param_groups"][0])
    assert sorted(state["state"]) == list(range(len(list(a.parameters())))) and set(state["state"][0]) == {"step", "exp_avg", "exp_avg_sq"}
    torch.save(dict(model_state_dict=a.state_dict(), optimizer_state_dict=state), tmp_path / "ck.pt")
    ck = torch.load(tmp_path / "ck.pt", map_location="cpu", weights_only=False)
    # continue with FusedAdam (a), with a stock Adam restored from the file (b), and with FusedAdam restored from
    # that stock Adam's own state_dict (c)
    b = _build(cfg, 2, dev); b.load_state_dict(ck["model_state_dict"])
    ob = torch.optim.Adam(b.parameters(), lr=1e-3, weight_decay=1e-4)
    ob.load_state_dict(ck["optimizer_state_dict"])
    c = _build(cfg, 2, dev); c.load_state_dict(ck["model_state_dict"])
    oc = snn.FusedAdam(c, lr=5e-2)
    oc.load_state_dict(ob.state_dict())
    assert oc.step_count == 3 and oc.param_groups[0]["lr"] == 1e-3 and oc.param_groups[0]["weight_decay"] == 1e-4
    run(a, oa, 2); run(b, ob, 2); run(c, oc, 2)
    fa, fb, fc = a.engine.flat, b.engine.flat, c.engine.flat
    # (c) is bit-identical; the stock Adam's update differs in the last bits, which the next bf16-operand forward/backward
    # amplifies (ReLU-mask flips) to a fraction of a percent of the 1e-3 update
    assert rel_l2(fb, fa) < 5e-4 and torch.equal(fc, fa)
    # a fresh optimizer has no per-parameter state, like torch's
    assert snn.FusedAdam(_build(cfg, 2, dev), lr=1e-3).state_dict()["state"] == {}
    bad = oa.state_dict()
    bad["state"][1]["exp_avg"] = torch.zeros(3)
    before = oc.exp_avg.clone()
    with pytest.raises(ValueError):
        oc.load_state_dict(bad)
    assert torch.equal(oc.exp_avg, before) and oc.step_count == 5


def test_loss_weight_zero_is_a_silent_participant(dev):
    """A rank without a batch of its own in a ragged last data-parallel step re-runs a batch with loss weight 0: its sum,
    its element count and its gradient are exactly zero, so the all-reduced global-batch loss ignores it."""
    import torch.distributed as dist
    from sres_b200 import nn as snn
    prd = torch.randn(3, 2, 16, 16, device=dev, requires_grad=True)
    tar = torch.randn(3, 2, 16, 16, device=dev)
    own = not dist.is_initialized()
    if own:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:29591", rank=0, world_size=1)
    try:
        for kind in ("l2", "charbonnier", "l1"):
            ref = snn.loss(prd, tar, kind)
            full = snn.loss(prd, tar, kind, dist.group.WORLD, 1.0)
            assert torch.equal(full, ref)
            prd.grad = None
            full.backward()
            assert prd.grad.abs().sum() > 0
    finally:
        if own:
            dist.destroy_process_group()
    prd.grad = None
    z = snn.loss(prd, tar, "l1", None, 0.0)      # no group: sum 0 over count 0
    z.backward()
    assert float(prd.grad.abs().sum()) == 0.0


def test_loss_decreases_when_training(dev):
    from sres_b200 import nn as snn
    cfg = O.model_cfg(nlayers=2, nblocks=2)
    torch.manual_seed(0)
    model = _build(cfg, 2, dev)
    opt = snn.FusedAdam(model, lr=2e-4)
    hr = synth_hr(8, 2, 96, smooth=True).to(dev)
    lr_in = snn.bicubic_resize(hr, 0.25)
    losses = []
    for _ in range(30):
        opt.zero_grad()
        loss = snn.loss(model(lr_in.requires_grad_(True)), hr, "l2")
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert np.isfinite(losses).all() and losses[-1] < 0.7 * losses[0]


def test_launch_accounting_is_counted_by_the_library(dev):
    """bench.py's `gpu_launches` comes from the library's own launch counter (sres_launch_count), read by the engine
    around its C calls.  Two residual groups of two RCABs, 48-px tiles: the fused two-convolution launches are in use, so a
    forward is head + 2 x (2 x (pair + channel attention) + group tail) + body tail + 4 + 4 up-convs + tail = 21 kernels
    once the packed weights are current, and a graph replay is credited with what its capture enqueued (that many plus
    the weight re-pack).  The counter moves by exactly what the engine reports."""
    from sres_b200 import nn as snn, _lib as L
    cfg = O.model_cfg(nlayers=2, nblocks=2)
    torch.manual_seed(0)
    model = _build(cfg, 2, dev)
    eng = model.engine
    hr = synth_hr(4, 2, 192, smooth=True).to(dev)
    lr_in = snn.bicubic_resize(hr, 0.25)
    lib = L.lib()
    counted = []
    for it in range(4):
        n0, e0 = lib.sres_launch_count(), eng.launches
        model.zero_grad()
        loss = snn.loss(model(lr_in.requires_grad_(True)), hr, "l2")
        fwd = eng.launches - e0
        loss.backward()
        torch.cuda.synchronize()
        counted.append((fwd, eng.launches - e0 - fwd, lib.sres_launch_count() - n0))
    if eng.use_graphs:
        assert counted[-1][0] == eng.launches_forward(48, 48) > 21        # a replay: the forward kernels + the weight re-pack
    else:
        assert all(f == 21 for f, _, _ in counted[1:])                    # packed weights are current after the first call
    assert counted[-1][1] == eng.launches_backward() > 0
    # what went through the library per iteration: the 4 loss kernels always; eager mode adds every forward and backward;
    # graph mode enqueues the forward twice in iteration 0 (eager call, then its capture), the backward eagerly in
    # iteration 0 and into its capture in iteration 1, and nothing but the loss afterwards (replays)
    f, b = counted[-1][0], counted[-1][1]
    through_lib = [c for _, _, c in counted]
    if eng.use_graphs:
        assert through_lib == [2 * f + b + 4, b + 4, 4, 4], counted
    else:
        assert through_lib[1:] == [f + b + 4] * 3, counted


def test_full_size_training_is_stable(dev):
    """RCAN-full x4 at the benchmark batch (64 tiles of 2x48x48), 40 optimiser steps on a fixed smooth batch through
    the graph-replayed path (side-stream weight gradients, PDL, fused Adam): the loss stays finite and goes down."""
    from sres_b200 import nn as snn
    torch.manual_seed(0)
    model = _build(O.model_cfg(cbottleneck=16), 2, dev)
    opt = snn.FusedAdam(model, lr=1e-4)
    hr = synth_hr(64, 2, 192, smooth=True).to(dev)
    lr_in = snn.bicubic_resize(hr, 0.25)
    losses = []
    for _ in range(40):
        opt.zero_grad()
        loss = snn.loss(model(lr_in.requires_grad_(True)), hr, "l2")
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert np.isfinite(losses).all() and losses[-1] < 0.8 * losses[0], losses[::8]
    assert torch.isfinite(model.engine.flat).all()


# ------------------------------------------------------------------------------------------------
# tiles: bit-exact
# ------------------------------------------------------------------------------------------------
def _tile_inputs(C, Y, X, seed, same_mask):
    var = synth_region(C, Y, X, seed)
    if C > 1 and same_mask:
        m = np.isnan(var[0])
        for v in var[1:]:
            v[np.isnan(v)] = 0.5
            v[m] = np.nan
    return var


def _dataset(C, tile, scale, order="reference", batch_size=7, region=None):
    from sres.base.util.config import ConfigContext
    from sres.data.batch import BatchDataset
    ConfigContext.deactivate()
    ConfigContext.set_defaults(task="SSS_SST-tiles-48" if C == 2 else "SST-tiles-48", dataset="synthetic_1200", platform="local")
    dfs = {2: [2], 4: [2, 2], 8: [2, 2, 2]}[scale]
    cc = ConfigContext.activate_global("sres", model="rcan-10-20-64", **{
        "task.batch_size": batch_size, "task.tile_size": dict(x=tile, y=tile), "task.tile_order": order,
        "model.downscale_factors": dfs, "model.nlayers": 1, "model.nblocks": 1})
    return cc, BatchDataset(region_source=(lambda t: region) if region is not None else None)


@pytest.mark.parametrize("name", [n for n in TILE_CASES if TILE_CASES[n][6]])
def test_tiles_extract_norm_flip_stitch_bit_exact(name, dev, golden_dir):
    from sres.base.util.config import ConfigContext
    C, Y, X, tile, scale, seed, same_mask = TILE_CASES[name]
    gold = np.load(os.path.join(golden_dir, f"tiles_{name}.npz"))
    var = _tile_inputs(C, Y, X, seed, same_mask)
    region = np.concatenate(var, 0)
    cc, ds = _dataset(C, tile, scale, region=region)
    try:
        ts = ds.load_timeslice(0)
        tiles_o, ids_o, gs_o = T.get_tiles(var, dict(x=tile, y=tile), scale)
        got = ts.values
        assert got.shape == tiles_o.shape and sha(got) == sha(tiles_o) == str(gold["tiles_sha"])      # bit-exact
        np.testing.assert_array_equal(ts.coords["tiles"], gold["tile_ids"])
        assert ts.attrs["grid_shape"] == gs_o
        # lnorm: floating point (mean/std reductions) -> tolerance; flips: exact permutations of it
        nb = ds.select_batch((7, 14))
        nb_o, st_o = T.lnorm(T.select_batch(tiles_o, 7, 14))
        np.testing.assert_allclose(nb.values, nb_o, rtol=0, atol=2e-5)
        np.testing.assert_allclose(nb.attrs["mean"].cpu().numpy(), st_o["mean"], rtol=1e-6)
        np.testing.assert_allclose(nb.attrs["std"].cpu().numpy(), st_o["std"], rtol=1e-5)
        base = nb.values
        for fi in range(8):
            fb = ds.norm(ts.data[7:14], (7, 14), fi)
            np.testing.assert_array_equal(fb.values, T.xyflip(base, fi))
        assert ds.select_batch((ts.shape[0], ts.shape[0] + 7)) is None
        assert list(ds.select_batch((ts.shape[0] - 3, ts.shape[0] + 4)).shape) == list(gold["last_batch_shape"])
        # stitching of raw tiles is bit-exact against the oracle AND against the reference's image hash
        from sres.controller.dual_trainer import ModelTrainer
        tr = object.__new__(ModelTrainer)
        tr.device = dev
        batches_o, batches_g = [], []
        for b in T.tile_batches(tiles_o.shape[0], 7):
            raw = T.select_batch(tiles_o, b["start"], b["end"])
            batches_o.append(dict(target=raw, input=np.ascontiguousarray(raw[:, :, ::scale, ::scale])))
            batches_g.append({k: torch.from_numpy(v).to(dev) for k, v in batches_o[-1].items()})
        for ivar in range(C):
            imgs_o = T.assemble_images(batches_o, ivar, ids_o, gs_o)
            imgs_g = tr.assemble_images(batches_g, ivar, ts.coords["tiles"], ts.attrs["grid_shape"])
            for k in imgs_o:
                assert imgs_g[k].dtype == imgs_o[k].dtype and sha(imgs_g[k]) == sha(imgs_o[k])
                assert int(np.isnan(imgs_g[k]).sum()) == int(gold[f"image_{ivar}_{k}_nan"])
                assert list(imgs_g[k].shape) == list(gold[f"image_{ivar}_{k}_shape"])
        # de-normalise + stitch (dual_trainer.py:67-77 + :449-480) fused in the stitch kernel: fed with the oracle's
        # normalised batches and statistics (pinned bit for bit to the reference, tests/test_oracle_golden.py) the images
        # must hash to the REFERENCE's images, dtype rule included
        nbatches, nstats = [], []
        for b in T.tile_batches(tiles_o.shape[0], 7):
            bd, st = T.lnorm(T.select_batch(tiles_o, b["start"], b["end"]))
            nbatches.append({"input": torch.from_numpy(np.ascontiguousarray(bd[:, :, ::scale, ::scale])).to(dev),
                             "target": torch.from_numpy(bd).to(dev)})
            nstats.append({k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in st.items()})
        for ivar in range(C):
            imgs = tr.assemble_images(nbatches, ivar, ts.coords["tiles"], ts.attrs["grid_shape"], nstats)
            for k, img in imgs.items():
                assert str(img.dtype) == str(gold[f"image_{ivar}_{k}_dtype"])
                assert sha(img) == str(gold[f"image_{ivar}_{k}_sha"]), (name, ivar, k)
    finally:
        ConfigContext.deactivate()


def test_tiles_reference_quirk_and_corrected_order(dev):
    from sres.base.util.config import ConfigContext
    C, Y, X, tile, scale, seed, same_mask = TILE_CASES["c2_diffmask"]
    var = _tile_inputs(C, Y, X, seed, same_mask)
    region = np.concatenate(var, 0)
    cc, ds = _dataset(C, tile, scale, order="reference", region=region)
    try:
        with pytest.raises(ValueError, match="cannot reshape"):
            ds.load_timeslice(0)
    finally:
        ConfigContext.deactivate()
    cc, ds = _dataset(C, tile, scale, order="corrected", region=region)
    try:
        ts = ds.load_timeslice(0)
        tiles_o, ids_o, _ = T.get_tiles(var, dict(x=tile, y=tile), scale, mode="corrected")
        assert sha(ts.values) == sha(tiles_o)
        np.testing.assert_array_equal(ts.coords["tiles"], ids_o)
    finally:
        ConfigContext.deactivate()


def test_full_size_region_roundtrip(dev):
    """Config 4 size: (1, 3000, 17280) region, 15 x 90 grid: stitch(extract(region)) reproduces the region
    bit for bit on surviving tiles and is NaN elsewhere (size-independent property, no oracle needed)."""
    from sres.base.util.config import ConfigContext
    from sres.controller.dual_trainer import ModelTrainer
    from sres.data.batch import synthetic_region
    region = synthetic_region(1, 3000, 17280, seed=5)
    cc, ds = _dataset(1, 48, 4, batch_size=64, region=region)
    try:
        ts = ds.load_timeslice(0)
        gs = ts.attrs["grid_shape"]
        assert gs == dict(x=90, y=15) and 0 < ts.shape[0] < 1350
        tr = object.__new__(ModelTrainer)
        tr.device = dev
        img = tr.assemble_images([dict(target=ts.data)], 0, ts.coords["tiles"], gs)["target"]
        crop = region[0, :15 * 192, :90 * 192]
        keep = np.zeros(1350, dtype=bool)
        keep[ts.coords["tiles"]] = True
        mask = np.repeat(np.repeat(keep.reshape(15, 90), 192, 0), 192, 1)
        assert np.array_equal(img[mask].astype(np.float32), crop[mask]) and np.isnan(img[~mask]).all()
        assert np.isfinite(crop[mask]).all()
    finally:
        ConfigContext.deactivate()


def test_llc4320_reader_bit_exact(dev, golden_dir, tmp_path):
    """The raw LLC4320 reader (pinned staging, gather index of the region built once from the template, one gather kernel per
    file) returns bit for bit what the reference's load_file + subset_roi return: against the oracle on the same files and
    against the reference's hashes, including -0.0 land points, NaNs inside the ocean, a region in the transposed / flipped
    western faces, time-index discovery and a data file that does not match the template."""
    from synth import LLC_CASES, synth_llc_files
    from sres.data.llc4320 import LLC4320Reader
    for name, (nx, roi, seed, land) in LLC_CASES.items():
        gold = np.load(os.path.join(golden_dir, f"llc_{name}.npz"))
        folder = str(tmp_path / name)
        files = synth_llc_files(folder, nx, seed, land)
        rd = LLC4320Reader(files["dataset_root"], files["dataset_files"], files["template"], roi, nx=nx, device=dev)
        assert rd.time_indices("V0") == [3, 4] and rd.time_indices("V1") == [3, 4]
        for v in range(2):
            for t in (3, 4):
                got = rd.load_file(f"V{v}", t).cpu().numpy()
                ref = T.llc_load_file(os.path.join(folder, files["template"]), rd.file_path(f"V{v}", t), nx, roi)
                assert got.shape == ref.shape and sha(got) == sha(np.ascontiguousarray(ref)) == str(gold[f"sha_V{v}_{t}"])
        assert rd.n_ocean == files["nocean"]
        reg = rd.load_region_data(["V0", "V1"], 4)
        assert reg.shape == (2,) + got.shape[1:] and sha(reg[1:].cpu().numpy()) == str(gold["sha_V1_4"])
        with open(rd.file_path("V0", 3), "ab") as fh:
            fh.write(b"\0\0\0\0")
        with pytest.raises(ValueError):
            rd.load_file("V0", 3)


def test_llc4320_source_feeds_the_tile_loader(dev, tmp_path):
    """`dataset.source: llc4320` through the mirrored BatchDataset: time indices from the files, tiles cut from the region the
    reader returns (device-resident end to end) equal the oracle's tiles of the oracle-read region."""
    from synth import synth_llc_files
    from sres.base.util.config import ConfigContext
    from sres.data.batch import BatchDataset
    nx, roi = 40, dict(y0=8, ys=100, x0=3, xs=150)
    files = synth_llc_files(str(tmp_path), nx, 31, 0.02, nvars=1)
    ConfigContext.deactivate()
    ConfigContext.set_defaults(task="SST-tiles-48", dataset="synthetic_1200", platform="local")
    ConfigContext.activate_global("sres", model="rcan-10-20-64", **{
        "task.tile_size": dict(x=12, y=12), "task.input_variables": dict(V0="v"), "task.target_variables": ["V0"],
        "dataset.source": "llc4320", "dataset.dataset_root": files["dataset_root"], "dataset.dataset_files": files["dataset_files"],
        "dataset.template": files["template"], "dataset.roi": roi, "dataset.nx": nx})
    try:
        ds = BatchDataset()
        assert ds.get_dset_time_indices() == [3, 4]
        ts = ds.load_timeslice(4)
        ref = T.llc_load_file(os.path.join(str(tmp_path), files["template"]), os.path.join(str(tmp_path), "raw/V0/V0.0004.shrunk"), nx, roi)
        tiles_o, ids_o, gs_o = T.get_tiles([ref], dict(x=12, y=12), 4)
        assert ts.attrs["grid_shape"] == gs_o and sha(ts.values) == sha(tiles_o)
        np.testing.assert_array_equal(ts.coords["tiles"], ids_o)
    finally:
        ConfigContext.deactivate()


# ------------------------------------------------------------------------------------------------
# the mirror of the reference controller API, end to end
# ------------------------------------------------------------------------------------------------
def test_controller_api_train_and_infer(dev, tmp_path):
    from sres.base.util.config import ConfigContext, cfg
    from sres.controller.config import ResultStructure, TSet
    from sres.controller.workflow import WorkflowController
    ConfigContext.deactivate()
    random.seed(3)
    wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local"), seed=1)
    wc.initialize("sres", "rcan-10-20-64", **{
        "model.nlayers": 2, "model.nblocks": 2, "task.batch_size": 8, "task.lr": 2e-4, "task.tile_size": dict(x=12, y=12),
        "task.tile_order": "corrected", "dataset.region": dict(ys=480, xs=480), "dataset.ntimes": 4,
        "task.ttsplit": dict(train=0.75, valid=0.25, test=0.0), "platform.results": str(tmp_path)})
    try:
        tr = wc.trainer
        assert type(tr.model).__module__ == "sres.model.rcan.network" and cfg().task.training_version.startswith("sres-rcan")
        first = tr.train(2, True, seed=4456, interp_loss=True, verbose=False)
        again = tr.train(1, False, seed=4456, interp_loss=True, verbose=False)   # resumes from the checkpoint
        assert np.isfinite(first["prediction"]) and np.isfinite(again["prediction"])
        assert os.path.exists(tr.checkpoint_manager.checkpoint_path(TSet.Train))
        ck = torch.load(tr.checkpoint_manager.checkpoint_path(TSet.Train), map_location="cpu", weights_only=False)
        assert set(ck) == {"epoch", "itime", "model_state_dict", "optimizer_state_dict", "loss"}
        assert list(ck["model_state_dict"].keys()) == list(O.param_shapes(O.model_cfg(nlayers=2, nblocks=2), 2, 2).keys())
        images, losses = wc.inference(0, ResultStructure.Image)
        assert set(images) == {"SSS", "SST"}
        for v in images:
            assert set(images[v]) == {"input", "target", "interpolated", "model"}
            assert images[v]["target"].shape == (480 // 48 * 48, 480 // 48 * 48) and images[v]["input"].shape == (120, 120)
            assert np.isfinite(losses[v]["model"]) and losses[v]["interpolated"] > 0
        # the epoch-end validation passes of train() kept a history and wrote the best-validation checkpoint
        hist = tr.eval_history[TSet.Validation]
        assert [h["epoch"] for h in hist] == [1, 1] and all(np.isfinite(h["model"]) for h in hist)
        vpath = tr.checkpoint_manager.checkpoint_path(TSet.Validation)
        assert os.path.exists(vpath)
        vck = torch.load(vpath, map_location="cpu", weights_only=False)
        assert abs(vck["loss"] - min(h["model"] for h in hist)) < 1e-9 and vck["loss"] == tr.validation_loss
        res, l2 = tr.evaluate(TSet.Validation, time_index=0)
        assert res["model"].shape[1:] == (2, 48, 48) and np.isfinite(l2["model"])
    finally:
        ConfigContext.deactivate()


def test_train_stream_equals_step_by_step(dev, tmp_path):
    """ModelTrainer.train_stream (host batches in, the next batch's copy issued under the running step) walks exactly the
    same optimizer steps as train_step batch by batch: identical losses and identical weights afterwards."""
    from sres.base.util.config import ConfigContext
    from sres.controller.workflow import WorkflowController
    ConfigContext.deactivate()
    over = {"model.nlayers": 2, "model.nblocks": 2, "task.batch_size": 6, "task.lr": 3e-4, "task.tile_size": dict(x=12, y=12),
            "dataset.region": dict(ys=480, xs=480), "dataset.ntimes": 2, "platform.results": str(tmp_path)}
    host = [synth_hr(6, 2, 48, seed=20 + i).pin_memory() for i in range(5)]
    try:
        out = []
        for mode in range(2):
            random.seed(3)
            wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local"), seed=1)
            wc.initialize("sres", "rcan-10-20-64", **over)
            tr = wc.trainer
            tr.model.train()
            if mode == 0:
                w0 = tr.model.engine.flat.detach().clone()
            else:                      # same initial weights as the first trainer (each draws its own from torch's RNG)
                tr.model.engine.flat.copy_(w0)
                tr.model.engine.mark_params_changed()
            if mode == 0:
                losses = [tr.train_step(h.to(dev)).item() for h in host]
            else:
                losses = [l.item() for l in tr.train_stream(iter(host))]
                assert list(tr.train_stream(iter([]))) == []
            out.append((losses, tr.model.engine.flat.detach().clone()))
            ConfigContext.deactivate()
        assert out[0][0] == out[1][0] and all(np.isfinite(out[0][0]))
        assert torch.equal(out[0][1], out[1][1])
    finally:
        ConfigContext.deactivate()


def test_edsr_through_the_controller_and_segments(dev, tmp_path):
    """EDSR (SURVEY 8f rank 3) through the mirrored factory / trainer: `model: edsr` picks sres.model.edsr.network,
    state_dict keys are the reference's, training runs and checkpoints, backward splits into 3 DP segments."""
    from sres.base.util.config import ConfigContext
    from sres.controller.workflow import WorkflowController
    from sres.controller.dual_trainer import TSet
    from sres_b200 import nn as snn
    wc = WorkflowController("sres", dict(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local"), seed=1)
    wc.initialize("sres", "edsr", **{
        "model.nlayers": 3, "model.res_scale": 0.5, "task.batch_size": 8, "task.lr": 2e-4, "task.tile_size": dict(x=12, y=12),
        "task.tile_order": "corrected", "dataset.region": dict(ys=480, xs=480), "dataset.ntimes": 2,
        "task.ttsplit": dict(train=0.5, valid=0.5, test=0.0), "platform.results": str(tmp_path)})
    try:
        tr = wc.trainer
        assert type(tr.model).__module__ == "sres.model.edsr.network"
        cfg_o = O.model_cfg(name="edsr", nlayers=3, res_scale=0.5)
        assert list(tr.model.state_dict().keys()) == list(O.param_shapes(cfg_o, 2, 2).keys())
        assert tr.model.engine.num_segments() == 3
        spans = [tr.model.engine.segment_params(i) for i in range(3)]
        assert sorted(spans)[0][0] == 0 and sum(c for _, c in spans) == tr.model.engine.n_params
        out = tr.train(2, True, seed=4456, interp_loss=True, verbose=False)
        assert np.isfinite(out["prediction"])
        assert os.path.exists(tr.checkpoint_manager.checkpoint_path(TSet.Train))
        # segment-wise backward == whole backward
        m = tr.model
        x = torch.randn(4, 2, 12, 12, device=dev)
        tgt = torch.randn(4, 2, 48, 48, device=dev)
        for p in m.parameters():
            p.grad = None
        snn.loss(m(x.clone().requires_grad_(True)), tgt, "l2").backward()
        whole = m.engine.flat_grad.clone()
        m.engine.flat_grad.zero_()
        prd = m(x.clone().requires_grad_(True))
        pr = prd.detach().requires_grad_(True)
        snn.loss(pr, tgt, "l2").backward()
        for seg in range(3):
            m.engine.backward(x, pr.grad.contiguous(), accumulate=False, seg_begin=seg, seg_end=seg + 1)
        assert torch.equal(m.engine.flat_grad, whole)
    finally:
        ConfigContext.deactivate()
