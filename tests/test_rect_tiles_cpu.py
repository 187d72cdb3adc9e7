"""CPU-only checks for rectangular tiles (task.tile_size {x, y} with x != y): the rectangular tile entry points are
exported and refuse malformed arguments before anything is launched, TileGrid matches the oracle per axis, and the
data-parallel row gather carries (C, sy, sx) rows."""
import ctypes as C
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
RECT = ("sres_tiles_finite_flags_hw", "sres_tiles_gather_hw", "sres_tiles_lnorm_hw", "sres_tiles_stitch_hw")


@pytest.fixture(scope="module")
def lib():
    from sres_b200 import _lib as L
    lib = L.lib()
    lib.sres_last_error.restype = C.c_char_p
    return lib


def test_rect_entry_points_declared_and_exported(lib):
    text = open(os.path.join(ROOT, "include", "sres_b200.h")).read()
    for n in RECT:
        assert f"{n}(" in text and hasattr(lib, n), n
    assert lib.sres_abi_version() == 4


def test_rect_entry_points_reject_bad_arguments(lib):
    """Every call below returns SRES_ERR_INVALID_ARG without touching the device (the pointers are never dereferenced)."""
    p = C.c_void_p(16)
    # region (2, 100, 120), grid 3 x 4 of 20 x 30 tiles at (y0, x0) = (10, 0) fits exactly on both axes
    Cc, Y, X, y0, x0, gy, gx = 2, 100, 120, 10, 0, 3, 4
    bad_geometry = [(0, 30, y0, x0), (20, 0, y0, x0), (-20, 30, y0, x0), (20, -30, y0, x0),
                    (31, 30, y0, x0),      # rows: 10 + 3 * 31 > 100
                    (20, 31, y0, x0),      # columns: 0 + 4 * 31 > 120
                    (20, 30, 41, x0),      # rows: 41 + 3 * 20 > 100
                    (20, 30, y0, 1)]       # columns: 1 + 4 * 30 > 120
    for Th, Tw, yy, xx in bad_geometry:
        assert lib.sres_tiles_finite_flags_hw(p, Cc, Y, X, yy, xx, Th, Tw, gy, gx, p, None) == 1, (Th, Tw, yy, xx)
        assert b"grid exceeds region" in lib.sres_last_error()
        assert lib.sres_tiles_gather_hw(p, Cc, Y, X, yy, xx, Th, Tw, gy, gx, p, 4, p, None) == 1, (Th, Tw, yy, xx)
        assert b"grid exceeds region" in lib.sres_last_error()
    # (the square entry points share the check: T = 31 overruns the rows of this grid)
    assert lib.sres_tiles_gather(p, Cc, Y, X, y0, x0, 31, gy, gx, p, 4, p, None) == 1
    for Th, Tw, flip in ((0, 30, 0), (20, 0, 0), (-1, 30, 0), (20, 30, -1), (20, 30, 8)):
        assert lib.sres_tiles_lnorm_hw(p, 6, Th, Tw, flip, C.c_void_p(32), p, p, None) == 1, (Th, Tw, flip)
        assert b"bad argument" in lib.sres_last_error()
    for flip in range(1, 8):                 # in place only without a flip (flips 4-7 also change the plane's shape)
        assert lib.sres_tiles_lnorm_hw(p, 6, 20, 30, flip, p, p, p, None) == 1, flip
        assert b"in-place" in lib.sres_last_error()
    for th, tw, ivar in ((0, 30, 0), (20, 0, 0), (20, -30, 0), (20, 30, 2), (20, 30, -1)):
        assert lib.sres_tiles_stitch_hw(p, Cc, ivar, th, tw, gy, gx, p, None, None, p, None) == 1, (th, tw, ivar)
        assert b"bad argument" in lib.sres_last_error()
    assert lib.sres_tiles_stitch_hw(p, Cc, 0, 20, 30, gy, gx, p, p, None, p, None) == 1      # mean without std


@pytest.mark.parametrize("tile,grid,origin", [
    (dict(x=12, y=7), dict(x=-1, y=-1), dict(x=0, y=0)),
    (dict(x=7, y=12), dict(x=-1, y=-1), dict(x=0, y=0)),
    (dict(x=12, y=50), dict(x=-1, y=-1), dict(x=0, y=0)),
    (dict(x=12, y=7), dict(x=5, y=-1), dict(x=40, y=3)),
    (dict(x=7, y=12), dict(x=-1, y=2), dict(x=0, y=17)),
])
def test_tile_grid_matches_oracle_per_axis(tile, grid, origin):
    import tiles_oracle as T
    from sres.base.util.config import ConfigContext
    from sres.data.tiles import TileGrid
    ConfigContext.deactivate()
    ConfigContext.set_defaults(task="SST-tiles-48", dataset="synthetic_1200", platform="local")
    try:
        with ConfigContext("sres", model="rcan-10-20-64", **{"task.tile_size": tile, "task.tile_grid": grid,
                                                            "task.origin": origin}):
            for shape in (dict(x=1200, y=1200), dict(x=1423, y=1000), dict(x=17280, y=3000)):
                g = TileGrid()
                gs = T.grid_shape(shape, tile, 4, grid)
                assert g.get_full_tile_size() == dict(x=tile["x"] * 4, y=tile["y"] * 4)
                assert g.get_grid_shape(image_shape=shape) == gs
                assert g.get_active_region(image_shape=shape) == T.active_region(origin, tile, 4, gs)
        # 200-row HR tiles (y: 50 at x4) cover all 3000 rows of the SWOT ROI
        with ConfigContext("sres", model="rcan-10-20-64", **{"task.tile_size": dict(x=48, y=50)}):
            roi = TileGrid().get_active_region(image_shape=dict(x=17280, y=3000))
            assert roi == dict(y=(0, 3000), x=(0, 17280))
    finally:
        ConfigContext.deactivate()


def _gather_worker(rank, world, port, out_q):
    sys.path.insert(0, os.path.join(ROOT, "super-resolution-climate_b200"))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from sres_b200.parallel import gather_rows
        rows = torch.arange(9 * 2 * 7 * 12, dtype=torch.float32).reshape(9, 2, 7, 12)
        counts = [5, 4]
        lo = sum(counts[:rank])
        ok = bool(torch.equal(gather_rows(rows[lo:lo + counts[rank]], counts, (2, 7, 12), torch.device("cpu")), rows))
        tr = rows.transpose(-1, -2).contiguous()           # the other orientation: (C, sx, sy) rows
        ok = ok and bool(torch.equal(gather_rows(tr[lo:lo + counts[rank]], counts, (2, 12, 7), torch.device("cpu")), tr))
        out_q.put((rank, ok))
    finally:
        dist.destroy_process_group()


def test_gather_rows_with_rectangular_rows():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(r[0] for r in res) == [0, 1] and all(r[1] for r in res), res
