"""torch.nn surface of the CUDA engine: an nn.Module with the reference RCAN's parameter names whose
forward/backward are single C-ABI calls, CUDA losses, resize (bicubic and the other interpolation modes) and a fused
flat Adam.

Reference interface mirrored here:
  RCAN / get_model            sres/model/rcan/network.py:5-27
  FModule.load_state_dict     sres/model/common/common.py:50-71 (tolerant of `tail.*` shape mismatches)
  l2loss                      sres/controller/stats.py:5-8
  charbonnier                 sres/controller/dual_trainer.py:196-198
  downsample / upsample       sres/base/util/array.py:72-76, 84-87
  torch.optim.Adam usage      sres/controller/dual_trainer.py:126, 310, 323
"""
import ctypes as C
import math
from typing import Any, Dict, Iterable, Mapping, Optional

import torch
import torch.nn as nn

from . import _lib as L
from .engine import RcanEngine

LOSS_KINDS = {"l2": 0, "charbonnier": 1, "l1": 2}


# ---------------------------------------------------------------------------------------------
# parameter holders that reproduce the reference module tree (and so its state_dict keys)
# ---------------------------------------------------------------------------------------------
class _ConvParams(nn.Module):
    """Holds `weight` / `bias` of one nn.Conv2d of the reference; the math runs in the engine."""

    def __init__(self, weight: torch.Tensor, bias: torch.Tensor):
        super().__init__()
        self.weight = nn.Parameter(weight)
        self.bias = nn.Parameter(bias)

    def forward(self, *a, **k):
        raise RuntimeError("sres_b200: layers are not callable one by one; call the RCAN module")


class _Holder(nn.Module):
    def forward(self, *a, **k):
        raise RuntimeError("sres_b200: layers are not callable one by one; call the RCAN module")


def _seq(mods):
    s = nn.Sequential()
    for i, m in mods:
        s.add_module(str(i), m)
    return s


class _RcanFunction(torch.autograd.Function):
    """forward = sres_rcan_forward, backward = sres_rcan_backward.  Parameter gradients are written
    into the engine's flat gradient buffer and exposed as `.grad` views (no per-tensor autograd
    accumulation: 1630 AccumulateGrad nodes would cost more than the GPU step)."""

    @staticmethod
    def forward(ctx, x, anchor, module):
        eng = module.engine
        xin = x.detach().contiguous().float()
        out = eng.forward(xin, training=True)
        ctx.module = module
        ctx.generation = eng.forward_generation(xin.shape[0], xin.shape[2], xin.shape[3])
        ctx.save_for_backward(xin)
        return out

    @staticmethod
    def backward(ctx, dout):
        module = ctx.module
        (xin,) = ctx.saved_tensors
        if ctx.generation != module.engine.forward_generation(xin.shape[0], xin.shape[2], xin.shape[3]):
            raise L.SresError("backward through a stale RCAN forward: the activation workspace holds one forward per "
                              "batch shape -- call backward before the next forward of the same shape")
        module._run_backward(xin, dout.contiguous().float())
        return None, None, None


def _resolve_device(device):
    device = torch.device(device if device is not None else "cuda")
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


class _EngineModule(nn.Module):
    """Shared plumbing of the engine-backed models: parameters are views into the engine's flat buffer under the
    reference's state_dict names; forward / backward are single C-ABI calls."""

    engine: RcanEngine

    def _finish_init(self, device):
        self._anchor = torch.zeros(1, device=device, requires_grad=True)
        self._grad_views: Dict[str, torch.Tensor] = {}
        self.ddp = None  # set by enable_data_parallel()
        self._build_tree()
        names = [k for k, _ in self.named_parameters()]
        assert names == [k for k, _ in self.engine.layout], "parameter order differs from the reference state_dict order"
        self._param_list = [p for _, p in self.named_parameters()]
        self.reset_parameters()

    def _views(self):
        eng = self.engine
        views, gviews, off = {}, {}, 0
        for name, shape in eng.layout:
            n = int(math.prod(shape))
            views[name] = eng.flat[off:off + n].view(shape)
            gviews[name] = eng.flat_grad[off:off + n].view(shape)
            off += n
        self._grad_views = gviews
        return views

    def _build_tree(self):
        raise NotImplementedError

    def reset_parameters(self):
        """nn.Conv2d's default init (kaiming_uniform(a=sqrt(5)) == U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for
        weight and bias), drawn on the host from torch's global RNG like the reference does."""
        eng = self.engine
        shapes = dict(eng.layout)
        host = torch.zeros(eng.n_padded)
        off = 0
        for name, shape in eng.layout:
            wshape = shape if name.endswith(".weight") else shapes[name[:-4] + "weight"]
            bound = 1.0 / math.sqrt(wshape[1] * wshape[2] * wshape[3])
            n = int(math.prod(shape))
            host[off:off + n] = (torch.rand(n) * 2 - 1) * bound
            off += n
        with torch.no_grad():
            eng.flat.copy_(host)
        eng.mark_params_changed()

    # -- nn.Module plumbing -----------------------------------------------------------------------
    def _apply(self, fn, recurse=True):
        probe = fn(torch.zeros(1, device=self.engine.device))
        if probe.device != self.engine.device or probe.dtype != torch.float32:
            raise L.SresError("sres_b200 RCAN lives on its CUDA device in fp32; build a new model to move it")
        return self

    def load_state_dict(self, state_dict: Mapping[str, Any], strict: bool = True, assign: bool = False):
        """Same tolerance as FModule.load_state_dict (common.py:50-71)."""
        own = self.state_dict()
        with torch.no_grad():
            for name, param in state_dict.items():
                if name in own:
                    try:
                        own[name].copy_(param.data if isinstance(param, nn.Parameter) else param)
                    except Exception:
                        if name.find("tail") >= 0:
                            print("Replace pre-trained upsampler to new one...")
                        else:
                            raise RuntimeError(f"While copying the parameter named {name}, whose dimensions in the model"
                                               f" are {own[name].size()} and whose dimensions in the checkpoint are {param.size()}.")
                elif strict and name.find("tail") == -1:
                    raise KeyError(f'unexpected key "{name}" in state_dict')
        if strict:
            missing = set(own.keys()) - set(state_dict.keys())
            if len(missing) > 0:
                raise KeyError(f'missing keys in state_dict: "{missing}"')
        self.engine.mark_params_changed()

    # -- forward / backward -----------------------------------------------------------------------
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if torch.is_grad_enabled():
            return _RcanFunction.apply(x, self._anchor, self)
        return self.engine.forward(x, training=False)

    def _run_backward(self, xin, dout):
        eng = self.engine
        plist = self._param_list
        first = plist[0].grad
        fresh = first is None
        if not fresh:
            gv = self._grad_views
            # accumulate in place only when every .grad is still our own view
            if first.data_ptr() != eng.flat_grad.data_ptr():
                raise L.SresError("RCAN parameters carry foreign .grad tensors; call optimizer.zero_grad() first")
        if self.ddp is None:
            eng.backward(xin, dout, accumulate=not fresh)
        else:
            self.ddp.backward(eng, xin, dout, accumulate=not fresh)
        if fresh:
            for (name, _), p in zip(eng.layout, plist):
                p.grad = self._grad_views[name]

    def enable_data_parallel(self, process_group=None, average: bool = False):
        """Overlap the per-segment gradient all-reduce (NCCL) with the rest of backward."""
        from .parallel import SegmentAllReduce
        self.ddp = SegmentAllReduce(self.engine, process_group, average)
        return self


class RCAN(_EngineModule):
    """Drop-in for the reference RCAN (sres/model/rcan/network.py:7-27): same constructor keywords
    (after hyper-parameter resolution), same parameter names/shapes, `model(x)` takes fp32
    (B,Cin,h,w) on the CUDA device and returns (B,Cout,h*s,w*s) taking part in autograd."""

    def __init__(self, nchannels_in=1, nchannels_out=1, nfeatures=64, nlayers=10, nblocks=20, cbottleneck=2,
                 kernel_size=3, bias=True, scale=4, device=None, **unused):
        super().__init__()
        if not bias:
            raise NotImplementedError("sres_b200 RCAN: bias=False is not supported")
        device = _resolve_device(device)
        self.parms = dict(nchannels_in=nchannels_in, nchannels_out=nchannels_out, nfeatures=nfeatures, nlayers=nlayers,
                          nblocks=nblocks, cbottleneck=cbottleneck, kernel_size=kernel_size, bias=bias, scale=scale)
        self.engine = RcanEngine(nchannels_in, nchannels_out, nfeatures, nlayers, nblocks, cbottleneck, scale, device)
        self._finish_init(device)

    # -- module tree ----------------------------------------------------------------------------
    def _build_tree(self):
        eng = self.engine
        views = self._views()

        def conv(prefix):
            return _ConvParams(views[prefix + ".weight"], views[prefix + ".bias"])

        G, R = eng.nlayers, eng.nblocks
        self.head = _seq([(0, conv("head.0"))])
        groups = []
        for g in range(G):
            blocks = []
            for r in range(R):
                pre = f"body.{g}.body.{r}.body"
                ca = _Holder()
                ca.conv_du = _seq([(0, conv(pre + ".3.conv_du.0")), (1, nn.ReLU(True)), (2, conv(pre + ".3.conv_du.2")),
                                   (3, nn.Sigmoid())])
                rcab = _Holder()
                rcab.body = _seq([(0, conv(pre + ".0")), (1, nn.ReLU(True)), (2, conv(pre + ".2")), (3, ca)])
                blocks.append((r, rcab))
            blocks.append((R, conv(f"body.{g}.body.{R}")))
            grp = _Holder()
            grp.body = _seq(blocks)
            groups.append((g, grp))
        groups.append((G, conv(f"body.{G}")))
        self.body = _seq(groups)
        ups = []
        for i, f in enumerate(eng.stages):
            ups.append((2 * i, conv(f"tail.0.{2 * i}")))
            ups.append((2 * i + 1, nn.PixelShuffle(f)))
        self.tail = _seq([(0, _seq(ups)), (1, conv("tail.1"))])


class EDSR(_EngineModule):
    """Drop-in for the reference EDSR (sres/model/edsr/network.py:9-32): head conv, `nlayers` ResBlocks
    (conv, ReLU, conv, *res_scale, +x; common/residual.py:30-54), conv, +head, SPUpsample, conv -- on the same
    tensor-core convolution kernels as RCAN.  batch_norm=True (never used by the shipped config) is not supported."""

    def __init__(self, nchannels_in=1, nchannels_out=1, nfeatures=64, nlayers=16, kernel_size=3, bias=True, scale=4,
                 res_scale=1.0, batch_norm=False, device=None, **unused):
        super().__init__()
        if not bias or batch_norm:
            raise NotImplementedError("sres_b200 EDSR: bias=False / batch_norm=True are not supported")
        device = _resolve_device(device)
        self.parms = dict(nchannels_in=nchannels_in, nchannels_out=nchannels_out, nfeatures=nfeatures, nlayers=nlayers,
                          kernel_size=kernel_size, bias=bias, scale=scale, res_scale=res_scale)
        self.engine = RcanEngine(nchannels_in, nchannels_out, nfeatures, 1, nlayers, 1, scale, device, arch="edsr",
                                 res_scale=res_scale)
        self._finish_init(device)

    def _build_tree(self):
        eng = self.engine
        views = self._views()

        def conv(prefix):
            return _ConvParams(views[prefix + ".weight"], views[prefix + ".bias"])

        R = eng.nblocks
        self.head = _seq([(0, conv("head.0"))])
        blocks = []
        for r in range(R):
            blk = _Holder()
            blk.body = _seq([(0, conv(f"body.{r}.body.0")), (1, nn.ReLU(True)), (2, conv(f"body.{r}.body.2"))])
            blocks.append((r, blk))
        blocks.append((R, conv(f"body.{R}")))
        self.body = _seq(blocks)
        ups = []
        for i, f in enumerate(eng.stages):
            ups.append((2 * i, conv(f"tail.0.{2 * i}")))
            ups.append((2 * i + 1, nn.PixelShuffle(f)))
        self.tail = _seq([(0, _seq(ups)), (1, conv("tail.1"))])


def get_model(**config) -> nn.Module:
    """Plugin entry point, same signature as sres/model/rcan/network.py:5-6."""
    return RCAN(**config)


def get_edsr_model(**config) -> nn.Module:
    """Plugin entry point of the EDSR family (sres/model/edsr/network.py:7-8)."""
    return EDSR(**config)


# ---------------------------------------------------------------------------------------------
# interpolation
# ---------------------------------------------------------------------------------------------
def bicubic_resize(t: torch.Tensor, scale_factor: float) -> torch.Tensor:
    """F.interpolate(t, scale_factor=scale_factor, mode='bicubic') on the CUDA kernel (no autograd)."""
    if t.device.type != "cuda":
        raise L.SresError("sres_b200.bicubic_resize needs a CUDA tensor")
    x = t.detach().contiguous().float()
    B, Cc, Hi, Wi = x.shape
    Ho, Wo = int(math.floor(Hi * scale_factor)), int(math.floor(Wi * scale_factor))
    out = torch.empty(B, Cc, Ho, Wo, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        L.check(L.lib().sres_bicubic_resize(L.ptr(x), L.ptr(out), B * Cc, Hi, Wi, Ho, Wo, C.c_double(1.0 / scale_factor),
                                            C.c_double(1.0 / scale_factor), L.cur_stream()), "sres_bicubic_resize")
    return out


def resize(t: torch.Tensor, scale_factor: float, mode: str) -> torch.Tensor:
    """F.interpolate(t, scale_factor=scale_factor, mode=mode) for 4-D input on the CUDA kernels (no autograd).
    mode: 'nearest', 'nearest-exact', 'bilinear', 'bicubic' or 'area' (align_corners=False, no antialias)."""
    if mode not in L.RESIZE_MODES:
        raise ValueError(f"sres_b200.resize: mode '{mode}' is not one of {', '.join(L.RESIZE_MODES)}")
    if t.device.type != "cuda":
        raise L.SresError("sres_b200.resize needs a CUDA tensor")
    x = t.detach().contiguous().float()
    B, Cc, Hi, Wi = x.shape
    Ho, Wo = int(math.floor(Hi * scale_factor)), int(math.floor(Wi * scale_factor))
    out = torch.empty(B, Cc, Ho, Wo, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        L.check(L.lib().sres_resize(L.ptr(x), L.ptr(out), B * Cc, Hi, Wi, Ho, Wo, 1.0 / scale_factor, 1.0 / scale_factor,
                                    L.RESIZE_MODES[mode], L.cur_stream()), "sres_resize")
    return out


# ---------------------------------------------------------------------------------------------
# losses
# ---------------------------------------------------------------------------------------------
class _LossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, prd, tar, kind, process_group, weight):
        lib = L.lib()
        p = prd.detach().contiguous().float()
        t = tar.detach().contiguous().float()
        B, Cc, H, W = p.shape
        tH, tW = t.shape[2], t.shape[3]
        if t.shape[0] != B or t.shape[1] != Cc or tH < H or tW < W:
            raise ValueError(f"loss: product {tuple(p.shape)} vs target {tuple(t.shape)}")
        lib.sres_loss_workspace_bytes.restype = C.c_size_t
        wsb = lib.sres_loss_workspace_bytes()
        with torch.cuda.device(p.device):
            ws = torch.empty(wsb, dtype=torch.uint8, device=p.device)
            stat = torch.zeros(2, dtype=torch.float64, device=p.device)
            loss = torch.empty(1, dtype=torch.float32, device=p.device)
            st = L.cur_stream()
            L.check(lib.sres_loss_sum(L.ptr(p), L.ptr(t), B * Cc, H, W, tH, tW, kind, L.ptr(stat), L.ptr(ws),
                                      C.c_size_t(wsb), st), "sres_loss_sum")
            if weight == 0.0:
                stat.zero_()      # a rank that only keeps the collectives company (ragged last global step)
            if process_group is not None:
                import torch.distributed as dist
                # global-batch loss (SURVEY.md 8e): the sum AND the element count are reduced, so the ranks may hold
                # batches of different sizes (the short last batch of a timeslice lands on an arbitrary rank)
                dist.all_reduce(stat, group=process_group)
            ntd = C.c_void_p(stat.data_ptr() + 8)
            L.check(lib.sres_loss_value(L.ptr(stat), C.c_double(0.0), ntd, kind, L.ptr(loss), st), "sres_loss_value")
        ctx.save_for_backward(p, t, loss, stat)
        ctx.kind, ctx.weight = kind, float(weight)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, gout):
        p, t, loss, stat = ctx.saved_tensors
        B, Cc, H, W = p.shape
        grad = torch.empty_like(p)
        gs = gout.detach().reshape(1).to(device=p.device, dtype=torch.float32).contiguous()  # no host sync
        with torch.cuda.device(p.device):
            L.check(L.lib().sres_loss_grad(L.ptr(p), L.ptr(t), B * Cc, H, W, t.shape[2], t.shape[3], ctx.kind, L.ptr(loss),
                                           C.c_double(0.0), C.c_void_p(stat.data_ptr() + 8), C.c_float(ctx.weight), L.ptr(gs),
                                           L.ptr(grad), L.cur_stream()),
                    "sres_loss_grad")
        return grad, None, None, None, None


def loss(prd: torch.Tensor, tar: torch.Tensor, kind: str = "l2", process_group=None, weight: float = 1.0) -> torch.Tensor:
    """Scalar loss on the CUDA kernels.  kind: 'l2' (RMSE over the whole batch tensor), 'charbonnier',
    'l1'.  With a process group the loss (and therefore the gradient) is that of the GLOBAL batch: per-rank sums and
    element counts are all-reduced, so ranks may hold batches of different sizes.  weight = 0 makes this rank a silent
    participant (its batch adds nothing to the sum, the count or the gradient) -- see parallel.dp_schedule."""
    if prd.device.type != "cuda":
        raise L.SresError("sres_b200.loss needs CUDA tensors")
    if weight not in (0.0, 1.0):
        raise ValueError("loss: weight must be 0 or 1")
    return _LossFunction.apply(prd, tar, LOSS_KINDS[kind], process_group, float(weight))


def l2loss(prd: torch.Tensor, tar: torch.Tensor, squared: bool = False) -> torch.Tensor:
    """Signature of sres/controller/stats.py:5-8."""
    out = loss(prd, tar, "l2")
    return out * out if squared else out


# ---------------------------------------------------------------------------------------------
# optimizer
# ---------------------------------------------------------------------------------------------
class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(lr, betas, eps, weight_decay) semantics as ONE kernel over the model's flat
    parameter buffer.  Same step()/zero_grad()/state_dict() surface the reference's trainer and
    CheckpointManager use (dual_trainer.py:126,310,323; checkpoints.py:20,44)."""

    def __init__(self, model: _EngineModule, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        if not isinstance(model, _EngineModule):
            raise TypeError("FusedAdam(model, ...): pass the sres_b200 RCAN / EDSR module (it owns the flat buffers)")
        super().__init__(list(model.parameters()), dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self.model = model
        eng = model.engine
        self.exp_avg = torch.zeros_like(eng.flat)
        self.exp_avg_sq = torch.zeros_like(eng.flat)
        self.step_count = 0

    @torch.no_grad()
    def step(self, closure=None):
        loss_v = closure() if closure is not None else None
        eng = self.model.engine
        if self.model._param_list[0].grad is None:
            return loss_v
        g = self.param_groups[0]
        self.step_count += 1
        with torch.cuda.device(eng.device):
            L.check(eng.lib.sres_adam_step_flat(L.ptr(eng.flat), L.ptr(eng.flat_grad), L.ptr(self.exp_avg),
                                                L.ptr(self.exp_avg_sq), C.c_int64(eng.n_padded), C.c_int64(self.step_count),
                                                C.c_double(g["lr"]), C.c_double(g["betas"][0]), C.c_double(g["betas"][1]),
                                                C.c_double(g["eps"]), C.c_double(g["weight_decay"]), L.cur_stream()),
                    "sres_adam_step_flat")
        eng.mark_params_changed()
        eng.launches += 1
        return loss_v

    def zero_grad(self, set_to_none: bool = True):
        if set_to_none:
            for p in self.model._param_list:
                p.grad = None
        else:
            self.model.engine.flat_grad.zero_()

    # -- torch.optim.Adam's state_dict layout ------------------------------------------------------------------------
    # {"state": {i: {"step", "exp_avg", "exp_avg_sq"}}, "param_groups": [{..., "params": [0..n-1]}]} with i the position of
    # the parameter in model.parameters() -- what the reference's CheckpointManager saves and loads
    # (sres/controller/checkpoints.py:20,44).  The flat moment buffers are cut along the engine's parameter layout.
    def _adam_group_template(self) -> Dict[str, Any]:
        probe = torch.optim.Adam([torch.zeros(1)], lr=1e-3)   # every key this torch version expects in a param group
        return {k: v for k, v in probe.state_dict()["param_groups"][0].items() if k != "params"}

    def state_dict(self):
        eng = self.model.engine
        g = dict(self._adam_group_template())
        g.update({k: v for k, v in self.param_groups[0].items() if k != "params"})
        state, off = {}, 0
        if self.step_count > 0:   # torch.optim.Adam has no per-parameter state before its first step
            for i, (_, shape) in enumerate(eng.layout):
                n = int(math.prod(shape))
                state[i] = dict(step=torch.tensor(float(self.step_count)),
                                exp_avg=self.exp_avg[off:off + n].view(shape).clone(),
                                exp_avg_sq=self.exp_avg_sq[off:off + n].view(shape).clone())
                off += n
        g["params"] = list(range(len(eng.layout)))
        return dict(state=state, param_groups=[g])

    def load_state_dict(self, sd):
        """Accepts torch.optim.Adam's layout (a reference checkpoint, or one of ours) and the flat private layout the
        first round of this build wrote ({step, exp_avg, exp_avg_sq, param_groups}).  Everything is checked before
        anything is modified."""
        eng = self.model.engine
        if "state" not in sd:   # round-1 private layout
            if not {"step", "exp_avg", "exp_avg_sq"} <= set(sd):
                raise ValueError("FusedAdam.load_state_dict: neither torch.optim.Adam's layout nor the flat layout")
            if sd["exp_avg"].numel() != self.exp_avg.numel():
                raise ValueError("FusedAdam.load_state_dict: flat moment buffers of another model")
            step, m_src, v_src = int(sd["step"]), [sd["exp_avg"]], [sd["exp_avg_sq"]]
            flat = True
        else:
            groups = sd["param_groups"]
            if len(groups) != 1 or list(groups[0].get("params", [])) != list(range(len(eng.layout))):
                raise ValueError("FusedAdam.load_state_dict: expected one param group over all "
                                 f"{len(eng.layout)} parameters in model order")
            if groups[0].get("amsgrad", False) or groups[0].get("maximize", False):
                raise ValueError("FusedAdam.load_state_dict: amsgrad / maximize are not supported")
            state = sd["state"]
            flat, m_src, v_src, steps = False, [], [], set()
            if state:
                for i, (name, shape) in enumerate(eng.layout):
                    st = state.get(i, state.get(str(i)))
                    if st is None or tuple(st["exp_avg"].shape) != tuple(shape) or tuple(st["exp_avg_sq"].shape) != tuple(shape):
                        raise ValueError(f"FusedAdam.load_state_dict: state of parameter {i} ({name}) is missing or has the wrong shape")
                    m_src.append(st["exp_avg"]); v_src.append(st["exp_avg_sq"])
                    steps.add(int(float(st["step"])))
                if len(steps) != 1:
                    raise ValueError("FusedAdam.load_state_dict: parameters carry different step counts")
            step = steps.pop() if state else 0
        with torch.no_grad():
            if not m_src:
                self.exp_avg.zero_(); self.exp_avg_sq.zero_()
            elif flat:
                self.exp_avg.copy_(m_src[0]); self.exp_avg_sq.copy_(v_src[0])
            else:
                off = 0
                for (_, shape), m, v in zip(eng.layout, m_src, v_src):
                    n = int(math.prod(shape))
                    self.exp_avg[off:off + n].copy_(m.reshape(-1)); self.exp_avg_sq[off:off + n].copy_(v.reshape(-1))
                    off += n
        self.step_count = step
        for g, saved in zip(self.param_groups, sd["param_groups"]):
            g.update({k: v for k, v in saved.items() if k in ("lr", "betas", "eps", "weight_decay")})
