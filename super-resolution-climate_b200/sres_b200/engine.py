"""Host-side engine over the C ABI: flat parameters, workspaces, forward/backward launches.

PyTorch is plumbing here (device memory, streams, torch.distributed); every FLOP of the hot path is
executed by libsres_b200.so.  There is no CPU or eager fallback: without a CUDA device or the built
library every entry point raises.
"""
import ctypes as C
import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib as L


class RcanDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("cin", C.c_int32), ("cout", C.c_int32), ("nfeatures", C.c_int32),
        ("n_groups", C.c_int32), ("n_blocks", C.c_int32), ("reduction", C.c_int32),
        ("n_up", C.c_int32), ("up_factor", C.c_int32 * 4),
        ("arch", C.c_int32), ("res_scale", C.c_float),
    ]


ARCH_RCAN, ARCH_EDSR = 0, 1


def upsampler_stages(scale: int) -> List[int]:
    """PixelShuffle factors of the reference Upsampler (sres/model/rcan/blocks.py:62-73)."""
    if scale >= 1 and scale & (scale - 1) == 0:
        return [2] * int(round(math.log2(scale)))
    if scale == 3:
        return [3]
    raise NotImplementedError(f"Upsampler: scale {scale}")  # blocks.py:74


def param_layout(nchannels_in: int, nchannels_out: int, nfeatures: int, nlayers: int, nblocks: int,
                 reduction: int, scale: int, kernel_size: int = 3):
    """Ordered [(state_dict key, shape)] of the reference RCAN (network.py:9-20) == flat-buffer order."""
    if kernel_size != 3:
        raise NotImplementedError("sres_b200 RCAN kernels are specialised for kernel_size == 3")
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin, k):
        out.append((name + ".weight", (cout, cin, k, k)))
        out.append((name + ".bias", (cout,)))

    Fn = nfeatures
    conv("head.0", Fn, nchannels_in, 3)
    for g in range(nlayers):
        for r in range(nblocks):
            pre = f"body.{g}.body.{r}.body"
            conv(pre + ".0", Fn, Fn, 3)
            conv(pre + ".2", Fn, Fn, 3)
            conv(pre + ".3.conv_du.0", Fn // reduction, Fn, 1)
            conv(pre + ".3.conv_du.2", Fn, Fn // reduction, 1)
        conv(f"body.{g}.body.{nblocks}", Fn, Fn, 3)
    conv(f"body.{nlayers}", Fn, Fn, 3)
    for i, f in enumerate(upsampler_stages(scale)):
        conv(f"tail.0.{2 * i}", f * f * Fn, Fn, 3)
    conv("tail.1", nchannels_out, Fn, 3)
    return out


def param_layout_edsr(nchannels_in: int, nchannels_out: int, nfeatures: int, nlayers: int, scale: int, kernel_size: int = 3):
    """Ordered [(state_dict key, shape)] of the reference EDSR (sres/model/edsr/network.py:14-26, ResBlock
    common/residual.py:41-46, SPUpsample common/upsample.py:44-46) == flat-buffer order."""
    if kernel_size != 3:
        raise NotImplementedError("sres_b200 EDSR kernels are specialised for kernel_size == 3")
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin, k):
        out.append((name + ".weight", (cout, cin, k, k)))
        out.append((name + ".bias", (cout,)))

    Fn = nfeatures
    conv("head.0", Fn, nchannels_in, 3)
    for r in range(nlayers):
        conv(f"body.{r}.body.0", Fn, Fn, 3)
        conv(f"body.{r}.body.2", Fn, Fn, 3)
    conv(f"body.{nlayers}", Fn, Fn, 3)
    for i, f in enumerate(upsampler_stages(scale)):
        conv(f"tail.0.{2 * i}", f * f * Fn, Fn, 3)
    conv("tail.1", nchannels_out, Fn, 3)
    return out


class RcanEngine:
    """One RCAN network on one GPU: owns the flat fp32 parameter / gradient buffers and per-shape
    workspaces, and issues the whole forward / backward kernel sequence with one C call each."""

    def __init__(self, nchannels_in: int, nchannels_out: int, nfeatures: int, nlayers: int, nblocks: int,
                 reduction: int, scale: int, device: torch.device, arch: str = "rcan", res_scale: float = 1.0):
        """arch 'rcan': nlayers residual groups of nblocks RCABs.  arch 'edsr': ONE group of `nblocks` ResBlocks
        (pass the reference's EDSR `nlayers` as nblocks and nlayers=1), no channel attention, `res_scale`."""
        device = torch.device(device)
        if arch not in ("rcan", "edsr"):
            raise ValueError(f"unknown arch {arch!r}")
        if arch == "edsr" and nlayers != 1:
            raise ValueError("EDSR engine: nlayers must be 1 (nblocks = number of ResBlocks)")
        self.arch, self.res_scale = arch, float(res_scale)
        if device.type != "cuda":
            raise L.SresError(f"sres_b200 RCAN needs a CUDA device (got {device}); there is no CPU fallback")
        self.lib = L.lib()
        self.device = device
        self.cin, self.cout, self.scale = nchannels_in, nchannels_out, scale
        self.nfeatures, self.nlayers, self.nblocks, self.reduction = nfeatures, nlayers, nblocks, reduction
        self.stages = upsampler_stages(scale)
        self.layout = (param_layout(nchannels_in, nchannels_out, nfeatures, nlayers, nblocks, reduction, scale) if arch == "rcan"
                       else param_layout_edsr(nchannels_in, nchannels_out, nfeatures, nblocks, scale))
        n = sum(int(math.prod(s)) for _, s in self.layout)
        d = self.desc(1, 8, 8)
        self.lib.sres_rcan_param_count.restype = C.c_int64
        n_c = self.lib.sres_rcan_param_count(C.byref(d))
        if n_c != n:
            L.check(1 if n_c < 0 else 0, "sres_rcan_param_count")
            raise L.SresError(f"parameter count mismatch: python {n}, library {n_c}")
        self.n_params = n
        self.n_padded = (n + 3) // 4 * 4
        with torch.cuda.device(device):
            self.flat = torch.zeros(self.n_padded, device=device, dtype=torch.float32)
            self.flat_grad = torch.zeros(self.n_padded, device=device, dtype=torch.float32)
        self._ws: Dict[Tuple[int, int, int, bool], torch.Tensor] = {}
        self._packed_version: Dict[Tuple[int, int, int, bool], int] = {}
        self._dirty_token = 0  # bumped by in-place updates torch cannot see (fused Adam)
        self.launches = 0      # kernels of ours enqueued so far (for bench accounting)
        self._fwd_count: Dict[tuple, int] = {}   # (B, H, W, training) -> kernels of one forward call (counted by the library)
        self._bwd_count: Dict[tuple, int] = {}   # ((B, H, W, True), seg_begin, seg_end) -> kernels of that backward call
        self._last_bwd_key = None
        # CUDA graphs: the whole forward (weight re-pack + ~640 kernels) and the whole backward (~1100
        # kernels) of a given batch shape are captured once and replayed -- static shapes, static workspace.
        self.use_graphs = os.environ.get("SRES_CUDA_GRAPHS", "1") != "0"
        self._l2_set = False
        # weight-gradient batches on a side stream (SRES_SIDE_STREAM=0 keeps everything on one stream)
        self._async = C.c_void_p(None)
        if os.environ.get("SRES_SIDE_STREAM", "1") != "0":
            with torch.cuda.device(device):
                L.check(self.lib.sres_async_create(C.byref(self._async)), "sres_async_create")
        self._graphs: Dict[tuple, dict] = {}
        self._fwd_generation: Dict[Tuple[int, int, int, bool], int] = {}

    # -- description / workspace --------------------------------------------------------------
    def desc(self, B: int, H: int, W: int) -> RcanDesc:
        d = RcanDesc()
        d.B, d.H, d.W = B, H, W
        d.cin, d.cout, d.nfeatures = self.cin, self.cout, self.nfeatures
        d.n_groups, d.n_blocks, d.reduction = self.nlayers, self.nblocks, self.reduction
        d.n_up = len(self.stages)
        for i, f in enumerate(self.stages):
            d.up_factor[i] = f
        d.arch = ARCH_EDSR if self.arch == "edsr" else ARCH_RCAN
        d.res_scale = self.res_scale
        return d

    MAX_SHAPES = 4   # shape entries (workspaces and their CUDA graphs) kept per engine; the least recently used is dropped

    @staticmethod
    def _shape_entry(key):
        """(B, H, W, training) and (B, W, H, training) are one cache entry: with rectangular tiles and xyflip a training
        epoch alternates between the two orientations, so they are kept and evicted together.  Each orientation still
        has its own workspace (the never-written padding rows of the gradient buffers differ between them)."""
        B, H, W, training = key
        return (B, min(H, W), max(H, W), training)

    def _evict_shapes(self, keep):
        """Ragged last batches and new inference shapes each need a multi-GB workspace: keep the MAX_SHAPES most recent
        shape entries."""
        keep_entry = self._shape_entry(keep)
        while len({self._shape_entry(k) for k in self._ws} | {keep_entry}) > self.MAX_SHAPES:
            old_entry = next(self._shape_entry(k) for k in self._ws if self._shape_entry(k) != keep_entry)
            torch.cuda.synchronize(self.device)
            for old in [k for k in self._ws if self._shape_entry(k) == old_entry]:
                for gk in [g for g in self._graphs if (g[1] == old if isinstance(g, tuple) and len(g) > 1 else False)]:
                    del self._graphs[gk]
                del self._ws[old]
                self._packed_version.pop(old, None)

    def workspace(self, B: int, H: int, W: int, training: bool) -> torch.Tensor:
        key = (B, H, W, training)
        ws = self._ws.get(key)
        if ws is not None:
            # most recently used last, together with the other orientation of its shape entry
            for k in [k for k in self._ws if self._shape_entry(k) == self._shape_entry(key)]:
                self._ws[k] = self._ws.pop(k)
        if ws is None:
            self._evict_shapes(key)
            nbytes = C.c_size_t(0)
            L.check(self.lib.sres_rcan_workspace_bytes(C.byref(self.desc(B, H, W)), int(training), C.byref(nbytes)),
                    "sres_rcan_workspace_bytes")
            with torch.cuda.device(self.device):
                ws = torch.zeros(nbytes.value, dtype=torch.uint8, device=self.device)  # zero-filled: see header
                if training and not self._l2_set:
                    # keep the fp32 trunk (read-modify-written by every RCAB) in the persisting part of L2 when it
                    # fits comfortably: measured +2.5 % on RCAN-full at B=64 (39 MB trunk, 48 MB set aside)
                    self._l2_set = True
                    env = os.environ.get("SRES_L2_PERSIST", "auto")
                    trunk_mb = (B * (H + 1) * (W + 1) * 256 + (1 << 20) - 1) >> 20
                    mb = (trunk_mb + 8 if trunk_mb <= 56 else 0) if env == "auto" else int(env)
                    if mb > 0:
                        L.check(self.lib.sres_l2_set_aside(C.c_size_t(mb << 20)), "sres_l2_set_aside")
            self._ws[key] = ws
        return ws

    def release_workspaces(self):
        self._graphs.clear()
        self._ws.clear()
        self._packed_version.clear()

    def mark_params_changed(self):
        self._dirty_token += 1

    def _version(self) -> int:
        return self.flat._version * 1000003 + self._dirty_token

    def _ensure_packed(self, key, ws, stream):
        v = self._version()
        if self._packed_version.get(key) != v:
            B, H, W, training = key
            L.check(self.lib.sres_rcan_pack_weights(C.byref(self.desc(B, H, W)), L.ptr(self.flat), L.ptr(ws),
                                                    int(training), stream), "sres_rcan_pack_weights")
            self._packed_version[key] = v

    # -- kernels launched per call (our claim for bench.py's gpu_launches) ----------------------
    # Counted, not derived: the library counts every kernel it enqueues (sres_launch_count, eager and stream-capture alike);
    # the engine reads the counter around each C call and remembers the number per (shape, segment range), so a graph
    # replay -- which does not pass through the library -- is credited with what its capture enqueued.
    def launches_forward(self, H: int, W: int, training: bool = True) -> int:
        """Kernels of one forward call at the most recently used batch size of this tile shape."""
        for key in reversed(list(self._fwd_count)):
            if key[1] == H and key[2] == W and key[3] == bool(training):
                return self._fwd_count[key]
        raise L.SresError("launches_forward: no forward of this shape has run yet")

    def launches_backward(self) -> int:
        """Kernels of one full backward pass (all segments) of the most recent backward shape."""
        key = self._last_bwd_key
        if key is None:
            raise L.SresError("launches_backward: no backward has run yet")
        nseg = self.num_segments()
        whole = self._bwd_count.get((key, 0, nseg))
        if whole is not None:
            return whole
        # the pass ran as several calls (data parallel: one per all-reduce bucket): chain the recorded ranges from segment 0
        total, s = 0, 0
        while s < nseg:
            ends = [e for (k, b, e) in self._bwd_count if k == key and b == s]
            if not ends:
                raise L.SresError(f"launches_backward: no backward call starting at segment {s} has run yet")
            e = max(ends)
            total += self._bwd_count[(key, s, e)]
            s = e
        return total

    # -- forward / backward ---------------------------------------------------------------------
    def _launch_forward(self, key, x, out, ws, always_pack=False):
        B, H, W, training = key
        st = L.cur_stream()
        n0 = self.lib.sres_launch_count()
        self._fwd_count.pop(key, None)   # most recently used last
        if always_pack:
            L.check(self.lib.sres_rcan_pack_weights(C.byref(self.desc(B, H, W)), L.ptr(self.flat), L.ptr(ws),
                                                    int(training), st), "sres_rcan_pack_weights")
        else:
            self._ensure_packed(key, ws, st)
        L.check(self.lib.sres_rcan_forward(C.byref(self.desc(B, H, W)), L.ptr(self.flat), L.ptr(x), L.ptr(out),
                                           L.ptr(ws), int(training), st), "sres_rcan_forward")
        self._fwd_count[key] = self.lib.sres_launch_count() - n0

    def forward(self, x: torch.Tensor, training: bool) -> torch.Tensor:
        if x.device != self.device:
            raise L.SresError(f"input on {x.device}, model on {self.device}")
        if x.dim() != 4 or x.shape[1] != self.cin:
            raise ValueError(f"expected (B,{self.cin},H,W) input, got {tuple(x.shape)}")
        x = x.detach().contiguous().float()
        B, _, H, W = x.shape
        key = (B, H, W, bool(training))
        sc = self.scale
        with torch.cuda.device(self.device):
            ws = self.workspace(*key)
            g = self._graphs.get(("fwd", key))
            if g is not None:
                g["x"].copy_(x)
                g["graph"].replay()
                out = g["out"].clone()
            else:
                out = torch.empty(B, self.cout, H * sc, W * sc, device=self.device, dtype=torch.float32)
                self._launch_forward(key, x, out, ws)
                if self.use_graphs:
                    # first call ran eagerly (lazy driver / attribute set-up happens outside capture); capture for the next ones
                    xs, outs = x.clone(), torch.empty_like(out)
                    graph = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize(self.device)
                    with torch.cuda.graph(graph):
                        self._launch_forward(key, xs, outs, ws, always_pack=True)
                    self._graphs[("fwd", key)] = dict(graph=graph, x=xs, out=outs)
        self._fwd_generation[key] = self._fwd_generation.get(key, 0) + 1
        self.launches += self._fwd_count[key]
        return out

    def forward_generation(self, B, H, W) -> int:
        return self._fwd_generation.get((B, H, W, True), 0)

    def num_segments(self) -> int:
        return self.nlayers + 2

    def segment_params(self, seg: int) -> Tuple[int, int]:
        off, cnt = C.c_int64(0), C.c_int64(0)
        L.check(self.lib.sres_rcan_segment_params(C.byref(self.desc(1, 8, 8)), seg, C.byref(off), C.byref(cnt)),
                "sres_rcan_segment_params")
        return off.value, cnt.value

    def _launch_backward(self, key, x, dout, accumulate, seg_begin, seg_end):
        B, H, W, _ = key
        n0 = self.lib.sres_launch_count()
        L.check(self.lib.sres_rcan_backward(C.byref(self.desc(B, H, W)), L.ptr(self.flat), L.ptr(x), L.ptr(dout),
                                            L.ptr(self.flat_grad), int(accumulate), L.ptr(self._ws[key]),
                                            seg_begin, seg_end, self._async, L.cur_stream()), "sres_rcan_backward")
        self._bwd_count[(key, seg_begin, seg_end)] = self.lib.sres_launch_count() - n0
        self._last_bwd_key = key

    def backward(self, x: torch.Tensor, dout: torch.Tensor, accumulate: bool, seg_begin: int = 0,
                 seg_end: Optional[int] = None):
        """Gradients of the flat parameter buffer into self.flat_grad for segments [seg_begin, seg_end).
        `x` must be the input of the most recent training-mode forward of this shape (its activations are
        what the workspace holds)."""
        B, _, H, W = x.shape
        key = (B, H, W, True)
        if key not in self._ws:
            raise L.SresError("backward without a matching training-mode forward")
        nseg = self.num_segments()
        seg_end = nseg if seg_end is None else seg_end
        whole = seg_begin == 0 and seg_end == nseg
        with torch.cuda.device(self.device):
            fg = self._graphs.get(("fwd", key))
            if self.use_graphs and fg is not None:
                # one graph per segment range; all ranges of a shape share the static dout / input buffers
                dk = ("dout", key)
                if dk not in self._graphs:
                    self._graphs[dk] = dict(dout=torch.empty_like(dout), token=None)
                slot = self._graphs[dk]
                douts = slot["dout"]
                # refresh the static copy whenever the caller's output gradient is a different tensor or has been modified
                # since the last copy (segments of one backward pass share it; a new pass always brings a new token)
                token = (dout.data_ptr(), dout._version, self._fwd_generation.get(key, 0))
                if slot["token"] != token:
                    douts.copy_(dout)
                    slot["token"] = token
                gk = ("bwd", key, bool(accumulate), seg_begin, seg_end)
                g = self._graphs.get(gk)
                if g is None:
                    # first call of this segment range runs eagerly (lazy module loading and kernel attributes stay outside
                    # capture, like forward); the second call captures
                    self._launch_backward(key, fg["x"], douts, accumulate, seg_begin, seg_end)
                    self._graphs[gk] = dict(graph=None)
                elif g["graph"] is None:
                    graph = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize(self.device)
                    with torch.cuda.graph(graph):
                        self._launch_backward(key, fg["x"], douts, accumulate, seg_begin, seg_end)
                    g["graph"] = graph
                    graph.replay()
                else:
                    g["graph"].replay()
            else:
                self._launch_backward(key, x, dout, accumulate, seg_begin, seg_end)
        if whole:
            self.launches += self.launches_backward()
