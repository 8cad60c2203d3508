"""Which kernel route each batch entry point takes, pinned by kernel-launch counts (Context.launches).

Launches per route:
  one-CTA tile kernel  1 per batch            grid mode   2 per pair (init + work kernel)
  naive kernel         1 per 4096 pairs       packing     3 (row planes, column planes, block summary)
  threshold pass       1                      window crop 1 (+1 to sanitise the pairs when a map index is given)
  merge table          1                      merge fold  1 per chunk
On a 1000 x 1000 map the automatic rule (set_grid_sweep(1)) takes grid mode for up to 4 pairs, the tile kernel
above.  A map too wide for the one-CTA kernel takes grid mode for up to 16 pairs, the naive kernel above.  The
`_dev` forms run after prepare_maps_dev (no packing), the host forms pack the maps once per call.  Every count is
taken after a warm-up call of the same kind, so that the 1/k table and the workspace already exist."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PACK = 3


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def new_ctx(vhp, naive=False):
    if not naive:
        return vhp.Context(0)
    old = os.environ.get("VHP_SWEEP_IMPL")
    os.environ["VHP_SWEEP_IMPL"] = "naive"
    try:
        return vhp.Context(0)
    finally:
        if old is None:
            del os.environ["VHP_SWEEP_IMPL"]
        else:
            os.environ["VHP_SWEEP_IMPL"] = old


@pytest.fixture(scope="module")
def ctx(vhp):
    c = new_ctx(vhp)
    yield c
    c.close()


def host_maps(nmaps, nx, ny, seed):
    g = np.random.default_rng(seed)
    return (g.random((nmaps, ny, nx)) > 0.05).astype(np.uint8)


def dev_maps(torch, nmaps, nx, ny, seed):
    return torch.from_numpy(host_maps(nmaps, nx, ny, seed)).cuda()


def sources(n, nx, ny, seed):
    g = np.random.default_rng(seed)
    return np.stack([g.integers(0, nx, n), g.integers(0, ny, n)], 1).astype(np.int32)


def launches_of(c, call):
    """launches of call() after one warm-up call"""
    call()
    c.synchronize()
    before = c.launches
    call()
    c.synchronize()
    return c.launches - before


def supported(vhp, nx, ny):
    lib = vhp.load_library()
    tile = getattr(lib, "_Z24vhp_sweep_tile_supportedii")
    grid = getattr(lib, "_Z24vhp_sweep_grid_supportedii")
    tile.restype = grid.restype = C.c_bool
    tile.argtypes = grid.argtypes = [C.c_int, C.c_int]
    return bool(tile(nx, ny)), bool(grid(nx, ny))


def sweep_dev_launches(torch, c, occ_t, n, seed=1):
    nmaps, ny, nx = occ_t.shape
    xy = torch.from_numpy(sources(n, nx, ny, seed)).cuda()
    out = torch.empty((n, ny, nx), dtype=torch.float32, device="cuda:0")
    c.prepare_maps_dev(occ_t)
    return launches_of(c, lambda: c.visibility_batch_dev(occ_t, xy, out))


@pytest.mark.parametrize("mode,n,want", [(1, 4, 8), (1, 5, 1), (0, 4, 1), (0, 5, 1), (2, 4, 8), (2, 5, 10)])
def test_sweep_dev(vhp, torch, ctx, mode, n, want):
    occ_t = dev_maps(torch, 1, 1000, 1000, 3)
    ctx.set_grid_sweep(mode)
    try:
        assert sweep_dev_launches(torch, ctx, occ_t, n) == want
    finally:
        ctx.set_grid_sweep(1)


@pytest.mark.parametrize("n", [4, 5])
def test_sweep_dev_naive(vhp, torch, n):
    c = new_ctx(vhp, naive=True)
    try:
        assert sweep_dev_launches(torch, c, dev_maps(torch, 1, 1000, 1000, 3), n) == 1
    finally:
        c.close()


@pytest.mark.parametrize("n,want", [(16, 32), (17, 1)])
def test_sweep_dev_too_wide_for_one_cta(vhp, torch, ctx, n, want):
    nx, ny = 12000, 64
    assert supported(vhp, nx, ny) == (False, True)
    assert sweep_dev_launches(torch, ctx, dev_maps(torch, 1, nx, ny, 4), n) == want


@pytest.mark.parametrize("thr,n,want", [(0.5, 5, 1), (0.0, 5, 2), (-1.0, 5, 2), (0.5, 4, 9)])
def test_bin_dev(vhp, torch, ctx, thr, n, want):
    occ_t = dev_maps(torch, 1, 1000, 1000, 5)
    xy = torch.from_numpy(sources(n, 1000, 1000, 6)).cuda()
    bits = torch.empty((n, 1000, 32), dtype=torch.int32, device="cuda:0")
    ctx.prepare_maps_dev(occ_t)
    assert launches_of(ctx, lambda: ctx.visibility_batch_bin_dev(occ_t, xy, thr, bits)) == want


@pytest.mark.parametrize("thr,nsrc,want", [(0.5, 5, 2), (0.0, 5, 3), (0.5, 4, 10)])
def test_merge_dev(vhp, torch, ctx, thr, nsrc, want):
    occ_t = dev_maps(torch, 1, 1000, 1000, 7)
    xy = torch.from_numpy(sources(nsrc, 1000, 1000, 8)).cuda()
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    vmax = torch.empty((1, 1000, 1000), dtype=torch.float32, device="cuda:0")
    ctx.prepare_maps_dev(occ_t)
    assert launches_of(ctx, lambda: ctx.visibility_merge_batch_dev(occ_t, xy, gptr, thr, vmax_t=vmax)) == want


@pytest.mark.parametrize("mode,with_map,want", [(1, False, 1), (1, True, 1), (2, False, 11), (2, True, 12)])
def test_window_dev(vhp, torch, ctx, mode, with_map, want):
    n, R = 5, 16
    occ_t = dev_maps(torch, 2, 1000, 1000, 9)
    xy = torch.from_numpy(sources(n, 1000, 1000, 10)).cuda()
    pm = torch.tensor([0, 1, 1, 0, 1], dtype=torch.int32, device="cuda:0") if with_map else None
    out = torch.empty((n, 2 * R + 1, 2 * R + 1), dtype=torch.float32, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        assert launches_of(ctx, lambda: ctx.visibility_window_batch_dev(occ_t, xy, R, out, src_map_t=pm)) == want
    finally:
        ctx.set_grid_sweep(1)


def test_host_forms(vhp, ctx):
    """each host call uploads the maps and packs them once (the sweep-based calls), or not at all"""
    occ = host_maps(1, 1000, 1000, 11)
    xy5, xy4 = sources(5, 1000, 1000, 12), sources(4, 1000, 1000, 13)
    assert launches_of(ctx, lambda: ctx.visibility_batch(occ, xy5, dtype=vhp.F32)) == PACK + 1
    assert launches_of(ctx, lambda: ctx.visibility_batch(occ, xy4, dtype=vhp.F32)) == PACK + 8
    assert launches_of(ctx, lambda: ctx.visibility_batch_bin(occ, xy5, 0.5)) == PACK + 1
    assert launches_of(ctx, lambda: ctx.visibility_batch_bin(occ, xy5, 0.0)) == PACK + 2
    assert launches_of(ctx, lambda: ctx.visibility_window_batch(occ, xy5, 16, dtype=vhp.F32)) == PACK + 1
    ctx.set_grid_sweep(2)
    try:
        assert launches_of(ctx, lambda: ctx.visibility_window_batch(occ, xy5, 16, dtype=vhp.F32)) == PACK + 11
    finally:
        ctx.set_grid_sweep(1)
    # fill + ray casting; the variants: one sweep kernel.  Neither reads the bit planes.
    assert launches_of(ctx, lambda: ctx.raycast_batch(occ, xy5, dtype=vhp.F32)) == 2
    assert launches_of(ctx, lambda: ctx.visibility_variant_batch(occ, xy5, vhp.VARIANT_QUEUE)) == 1


def test_planner_host_packs_under_naive(vhp):
    c = new_ctx(vhp, naive=True)
    try:
        c.set_grid_sweep(0)  # one persistent CTA per problem: one launch
        occ = host_maps(1, 101, 101, 14)
        occ[0, 5, 5] = occ[0, 95, 95] = 1
        assert launches_of(c, lambda: c.planner_batch(occ, [(5, 5, 95, 95)], max_iter=20)) == PACK + 1
    finally:
        c.close()


@pytest.mark.parametrize("mode,nx,y1,want", [(1, 1024, 1023, 1), (1, 1024, 1024, 2), (2, 1024, 1023, 2),
                                             (0, 1024, 1024, 1), (1, 12000, 64, 2)])
def test_strip_sweep(vhp, torch, ctx, mode, nx, y1, want):
    """vhp_strip_sweep_dev of rows [0, y1) from a source on row 0 (no halo rows): grid mode from 2^20 strip
    cells on in mode 1, always in mode 2, never in mode 0; always on a map too wide for one CTA"""
    ny = 1024 if nx == 1024 else 64
    occ_t = dev_maps(torch, 1, nx, ny, 15)
    out = torch.empty((y1, nx), dtype=torch.float64, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        call = lambda: ctx._check(ctx.lib.vhp_strip_sweep_dev(  # noqa: E731
            ctx.h, occ_t.data_ptr(), nx, ny, 5, 0, 0, y1, None, vhp.F64, out.data_ptr()))
        assert launches_of(ctx, call) == want
    finally:
        ctx.set_grid_sweep(1)


def test_strip_sweep_too_wide_without_grid_mode(vhp, torch, ctx):
    nx, ny = 12000, 64
    occ_t = dev_maps(torch, 1, nx, ny, 16)
    out = torch.empty((ny, nx), dtype=torch.float64, device="cuda:0")
    ctx.set_grid_sweep(0)
    try:
        st = ctx.lib.vhp_strip_sweep_dev(ctx.h, occ_t.data_ptr(), nx, ny, 5, 0, 0, ny, None, vhp.F64, out.data_ptr())
        assert st == -5  # VHP_ERR_UNSUPPORTED
    finally:
        ctx.set_grid_sweep(1)
