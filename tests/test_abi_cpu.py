"""CPU-only checks: the C-ABI library loads and exports every symbol include/sres_b200.h declares,
argument validation fails loudly, and the host-side mirror logic (config, tile iterators, source
tables, DP sharding) matches the oracle.  No compute calls (there is no GPU here)."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
HEADER = os.path.join(ROOT, "include", "sres_b200.h")


@pytest.fixture(scope="module")
def lib():
    from sres_b200 import _lib as L
    return L.lib()


def declared_symbols():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"SRES_API\s+[\w\s\*]+?\b(sres_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/sres_b200.h but not exported"
    assert lib.sres_abi_version() == 3


def test_header_cites_reference_lines():
    text = open(HEADER).read()
    for needle in ("network.py:22-27", "dual_trainer.py:557-571", "stats.py:5-8", "raw.py:216-233", "dual_trainer.py:449-480",
                   "cnn.py:8-9", "blocks.py"):
        assert needle in text


def test_geometry_helpers(lib):
    lib.sres_ptl_rows.restype = C.c_int64
    assert lib.sres_ptl_rows(64, 48, 48) == 64 * 49 * 49
    tr = lib.sres_conv_tile_rows(48, 48)
    assert tr in (126, 128)   # 126: three-taps-per-MMA kernel (tiles overlap by two rows)
    assert lib.sres_conv_mtiles(64, 48, 48) == (64 * 49 * 49 + tr - 1) // tr


def test_param_count_and_segments(lib):
    from sres_b200.engine import RcanDesc, param_layout
    d = RcanDesc()
    d.B, d.H, d.W, d.cin, d.cout, d.nfeatures, d.n_groups, d.n_blocks, d.reduction, d.n_up = 4, 48, 48, 2, 2, 64, 10, 20, 2, 2
    d.up_factor[0] = d.up_factor[1] = 2
    lib.sres_rcan_param_count.restype = C.c_int64
    n = lib.sres_rcan_param_count(C.byref(d))
    assert n == 16313602                                                       # SURVEY.md 3.2
    layout = param_layout(2, 2, 64, 10, 20, 2, 4)
    assert len(layout) == 1630 and sum(int(np.prod(s)) for _, s in layout) == n
    import rcan_oracle as O
    assert [k for k, _ in layout] == list(O.param_shapes(O.model_cfg(), 2, 2).keys())
    # the backward segments partition the flat parameter buffer
    nseg = lib.sres_rcan_num_segments(C.byref(d))
    assert nseg == 12
    spans = []
    for s in range(nseg):
        off, cnt = C.c_int64(), C.c_int64()
        assert lib.sres_rcan_segment_params(C.byref(d), s, C.byref(off), C.byref(cnt)) == 0
        spans.append((off.value, cnt.value))
    # the data-parallel all-reduce buckets (groups of consecutive segments) are contiguous parameter ranges, cover the buffer
    # once and are balanced: two buckets of RCAN-full split after the fifth residual group from the end
    from sres_b200.parallel import SegmentAllReduce
    for nb in (0, 1, 2, 3, 4, 12, 40):
        buckets = SegmentAllReduce._make_buckets(spans, nb)
        assert len(buckets) == (nseg if nb == 0 or nb >= nseg else nb)
        assert [b[0] for b in buckets] == [0] + [b[1] for b in buckets[:-1]] and buckets[-1][1] == nseg
        cover = sorted((off, cnt) for _, _, off, cnt in buckets)
        assert cover[0][0] == 0 and all(a[0] + a[1] == b[0] for a, b in zip(cover, cover[1:])) and cover[-1][0] + cover[-1][1] == n
    two = SegmentAllReduce._make_buckets(spans, 2)
    assert (two[0][0], two[0][1], two[1][1]) == (0, 6, 12) and abs(two[0][3] - two[1][3]) < 0.1 * n
    spans.sort()
    assert spans[0][0] == 0 and all(a[0] + a[1] == b[0] for a, b in zip(spans, spans[1:])) and spans[-1][0] + spans[-1][1] == n
    ws = C.c_size_t()
    assert lib.sres_rcan_workspace_bytes(C.byref(d), 1, C.byref(ws)) == 0 and ws.value > 0


def test_edsr_param_layout_and_segments(lib):
    """EDSR through the same C entry points (arch flag): parameter count / order equal the reference's state_dict
    (via the oracle's restatement), three backward segments partition the flat buffer, bad descriptions are refused."""
    from sres_b200.engine import ARCH_EDSR, RcanDesc, param_layout_edsr
    import rcan_oracle as O
    d = RcanDesc()
    d.B, d.H, d.W, d.cin, d.cout, d.nfeatures, d.n_groups, d.n_blocks, d.reduction, d.n_up = 4, 48, 48, 2, 2, 64, 1, 16, 1, 2
    d.up_factor[0] = d.up_factor[1] = 2
    d.arch, d.res_scale = ARCH_EDSR, 1.0
    lib.sres_rcan_param_count.restype = C.c_int64
    n = lib.sres_rcan_param_count(C.byref(d))
    layout = param_layout_edsr(2, 2, 64, 16, 4)
    shapes = O.param_shapes(O.model_cfg(name="edsr"), 2, 2)
    assert [k for k, _ in layout] == list(shapes.keys()) and [tuple(s_) for _, s_ in layout] == [tuple(v) for v in shapes.values()]
    assert n == sum(int(np.prod(s_)) for _, s_ in layout)
    assert lib.sres_rcan_num_segments(C.byref(d)) == 3
    spans = []
    for seg in range(3):
        off, cnt = C.c_int64(), C.c_int64()
        assert lib.sres_rcan_segment_params(C.byref(d), seg, C.byref(off), C.byref(cnt)) == 0
        spans.append((off.value, cnt.value))
    spans.sort()
    assert spans[0][0] == 0 and all(a[0] + a[1] == b[0] for a, b in zip(spans, spans[1:])) and spans[-1][0] + spans[-1][1] == n
    d.n_groups = 2
    assert lib.sres_rcan_param_count(C.byref(d)) < 0          # EDSR is one group of ResBlocks
    d.n_groups, d.res_scale = 1, 0.0
    assert lib.sres_rcan_param_count(C.byref(d)) < 0          # res_scale must be positive
    d.res_scale, d.arch = 1.0, 7
    assert lib.sres_rcan_param_count(C.byref(d)) < 0          # unknown architecture


def test_invalid_arguments_fail_loudly(lib):
    from sres_b200 import _lib as L
    from sres_b200.engine import RcanDesc
    lib.sres_last_error.restype = C.c_char_p
    d = RcanDesc()
    d.B, d.H, d.W, d.cin, d.cout, d.nfeatures, d.n_groups, d.n_blocks, d.reduction, d.n_up = 1, 8, 8, 2, 2, 32, 1, 1, 2, 0
    ws = C.c_size_t()
    assert lib.sres_rcan_workspace_bytes(C.byref(d), 0, C.byref(ws)) == 2      # SRES_ERR_UNSUPPORTED
    assert b"nfeatures" in lib.sres_last_error()
    assert lib.sres_conv3x3_igemm(None, None) == 1                              # SRES_ERR_INVALID_ARG
    with pytest.raises(L.SresError):
        L.check(lib.sres_pack_conv_weights(None, None, 0, 64, 64, 64, 1, 0, None), "pack")
    assert lib.sres_adam_step_flat(None, None, None, None, C.c_int64(8), C.c_int64(1), C.c_double(1e-3), C.c_double(0.9),
                                   C.c_double(0.999), C.c_double(1e-8), C.c_double(0.0), None) == 1
    # weight-gradient jobs whose output-channel mapping is malformed are refused before the device is touched (the
    # pointers are never dereferenced): oc_stride 0 would have 64 threads race on one element
    for cout_total, stride, offset in ((64, 0, 0), (64, -1, 0), (256, 4, 4), (256, 4, -1), (0, 1, 0), (-64, 1, 0)):
        job = L.WgradJob(16, 16, 16, 16, cout_total, stride, offset, 0, 1.0)
        assert lib.sres_conv3x3_wgrad_batch(C.byref(job), 1, 2, 8, 8, C.c_void_p(16), C.c_size_t(1 << 30), None) == 1
        assert b"oc_stride" in lib.sres_last_error(), (cout_total, stride, offset)
    good = L.WgradJob(16, 16, 16, 16, 256, 4, 3, 0, 1.0)
    bad = L.WgradJob(16, 16, 16, 16, 256, 4, 0, 0, 1.0)
    bad.oc_stride = 0
    jobs = (L.WgradJob * 2)(good, bad)                                          # the second job of a batch is checked too
    assert lib.sres_conv3x3_wgrad_batch(jobs, 2, 2, 8, 8, C.c_void_p(16), C.c_size_t(1 << 30), None) == 1
    assert lib.sres_conv3x3_wgrad(C.c_void_p(16), C.c_void_p(16), 2, 8, 8, C.c_void_p(16), None, 64, 0, 0, 0, C.c_void_p(16),
                                  C.c_size_t(1 << 30), None) == 1


def test_no_cpu_fallback():
    import torch
    from sres_b200 import _lib as L
    from sres_b200.engine import RcanEngine
    with pytest.raises(L.SresError):
        RcanEngine(2, 2, 64, 1, 1, 2, 4, torch.device("cpu"))
    # the product never imports the oracle
    pkg = os.path.join(ROOT, "super-resolution-climate_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "rcan_oracle" not in src and "tiles_oracle" not in src and "/root/reference" not in src, f


def test_config_and_tile_iterators_match_oracle():
    import tiles_oracle as T
    from sres.base.util.config import ConfigContext, cfg
    from sres.data.tiles import TileBatchIterator, TileGrid
    ConfigContext.set_defaults(task="SSS_SST-tiles-48", dataset="synthetic_1200", platform="local")
    with ConfigContext("sres", model="rcan-10-20-64", **{"task.batch_size": 7, "model.nlayers": 4}):
        assert cfg().model.nlayers == 4 and cfg().model.nblocks == 20 and cfg().task.batch_size == 7
        assert cfg().task.training_version == "sres-rcan-10-20-64-synthetic_1200-SSS_SST-tiles-48"
        random.seed(99)
        got = [b for b in TileBatchIterator(ntiles=29, randomize=True)]
        random.seed(99)
        assert got == T.tile_batches(29, 7, randomize=True)
        for shape in (dict(x=1200, y=1200), dict(x=1423, y=1000), dict(x=17280, y=3000)):
            g = TileGrid()
            assert g.get_grid_shape(image_shape=shape) == T.grid_shape(shape, dict(x=48, y=48), 4)
            assert g.get_active_region(image_shape=shape) == T.active_region(dict(x=0, y=0), dict(x=48, y=48), 4, T.grid_shape(shape, dict(x=48, y=48), 4))
    assert ConfigContext.cfg is None
    with pytest.raises(AssertionError):
        ConfigContext.activate_global("sres", model="rcan-10-20-64")
        ConfigContext("sres", model="rcan-10-20-64")
    ConfigContext.deactivate()


def test_source_table_matches_reference_order(golden_dir):
    """Host half of get_tiles: which candidate tile feeds slot (n,c) -- checked against the tile ids the
    unmodified reference produced (tests/golden/tiles_*.npz) and against the oracle's tiles."""
    import tiles_oracle as T
    from synth import TILE_CASES, synth_region
    from sres.data.batch import source_table
    for name in ("c1_1200", "c2_1200", "c1_odd"):
        Cn, Y, X, tile, scale, seed, same = TILE_CASES[name]
        gold = np.load(os.path.join(golden_dir, f"tiles_{name}.npz"))
        var = synth_region(Cn, Y, X, seed)
        if Cn > 1:
            m = np.isnan(var[0])
            for v in var[1:]:
                v[np.isnan(v)] = 0.5
                v[m] = np.nan
        region = np.concatenate(var, 0)
        gs = T.grid_shape(dict(x=X, y=Y), dict(x=tile, y=tile), scale)
        Tt = tile * scale
        cand = region[:, :gs["y"] * Tt, :gs["x"] * Tt].reshape(Cn, gs["y"], Tt, gs["x"], Tt).swapaxes(2, 3).reshape(-1, Tt, Tt)
        flags = np.isfinite(cand).all(axis=(1, 2)).astype(np.int32)
        src, ids = source_table(flags, Cn, gs["y"] * gs["x"], "reference")
        np.testing.assert_array_equal(ids, gold["tile_ids"])
        tiles, _, _ = T.get_tiles(var, dict(x=tile, y=tile), scale)
        np.testing.assert_array_equal(cand[src].reshape(tiles.shape), tiles)
    flags = np.array([1, 1, 1, 0, 1, 1], dtype=np.int32)          # 2 variables x 3 tiles, masks differ
    with pytest.raises(ValueError, match="cannot reshape"):
        source_table(flags, 2, 3, "reference")
    src, ids = source_table(flags, 2, 3, "corrected")
    assert list(ids) == [1, 2] and list(src) == [1, 4, 2, 5]


def test_shard_range_covers_everything():
    from sres_b200.parallel import shard_range
    for n in (0, 1, 7, 64, 1350):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
