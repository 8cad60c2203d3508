"""Every kernel route on both sides of its size limit, against the oracle.

The limits come from the library's predicates (test_limits_cpu: bisection over vhp_sweep_tile_supported,
vhp_planner_supported, vhp_sweep_window_supported and vhp_sweep_merge_view_supported), so these tests follow the
tile layout: each runs the largest shape a route takes, where its shared memory is all but full (at 9632 x 40 the
8-warp CTA leaves 16 bytes unused), and the first shape past it, which takes another route.  The route is pinned by
kernel-launch counts (test_gpu_routes).  The launch-grid limits are the 65 535 pairs of one ray-casting launch and
the 65 535 maps of one environment-generator launch; the largest side is 16384 (check_grid_dtype).  All
comparisons are exact: fp64 bit for bit, fp32 as the oracle's fp64 rounded once.

Run time on a B200 is dominated by the CPU oracle: about 20 s for the 16384^2 map, about 15 s for the 9472 x 1000
and 9473 x 1000 edge maps together, a few seconds for each of the other tests."""
import numpy as np
import pytest

from conftest import rect_map
from test_gpu_cover import expected as cover_expected, check as cover_check
from test_gpu_merge import check as merge_check, expected as merge_expected
from test_gpu_merge_range import expected as range_expected
from test_gpu_merge_view import expected as view_expected
from test_gpu_planner import check as planner_check
from test_gpu_routes import PACK, dev_maps, launches_of, new_ctx, supported
from test_limits_cpu import MAX_SIDE, planner_edge, predicates, tile_edge, view_edge, window_edge
from test_window_cpu import window_of

pytestmark = pytest.mark.gpu

EDGE_NYS = (40, 64, 65, 1000)
THR = 0.5
TILE_PAIRS = 17  # more than grid_max (at most 16): the automatic rule leaves grid mode


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def preds():
    return predicates()


def edge_sources(nx, ny):
    """corners, a tile border in the middle (x mod 32 = 31 and 0), the middle and x = 31 on row 0"""
    b = 32 * (nx // 64)
    s = [(0, 0), (nx - 1, ny - 1), (0, ny - 1), (nx - 1, 0), (b - 1, ny // 2), (b, ny - 1), (nx // 2 + 5, ny // 3),
         (31, 0)]
    return np.array([(min(max(x, 0), nx - 1), min(max(y, 0), ny - 1)) for x, y in s], np.int32)


_CASES = {}


def edge_case(oracle, nx, ny):
    """(occ, sources, oracle fields) of a random-rectangle map, cached for the module"""
    if (nx, ny) not in _CASES:
        occ = rect_map(nx, ny, max(1, nx * ny // 300), nx + 7 * ny, 1, 6)
        srcs = edge_sources(nx, ny)
        fields = np.stack([oracle.compute_visibility(occ, int(sx), int(sy)) for sx, sy in srcs])
        _CASES[(nx, ny)] = occ, srcs, fields
    return _CASES[(nx, ny)]


def launches_and_result(c, call):
    """launches of call() after one warm-up call (launches_of), and what the counted call returned"""
    out = {}

    def run():
        out["r"] = call()
    return launches_of(c, run), out["r"]


def f32(a):
    return a.astype(np.float32)


def check_fields(vhp, c, occ, xy, want, what):
    for dt in (vhp.F64, vhp.F32):
        got = c.visibility_batch(occ, xy, dtype=dt)
        assert np.array_equal(got, want if dt == vhp.F64 else f32(want)), (what, dt)


def check_bits_and_runs(vhp, c, occ, xy, want, what):
    """bits and row runs against the oracle field >= THR (padding bits of the last word included)"""
    nx = occ.shape[-1]
    want_bits = vhp.pack_bits(want >= THR)
    assert np.array_equal(c.visibility_batch_bin(occ, xy, THR), want_bits), what
    rc, pp, tr = c.visibility_batch_runs(occ, xy, THR)
    assert np.array_equal(vhp.runs_to_bits(rc, pp, tr, nx), want_bits), what


# ---- one-CTA tile kernel: the width edge -------------------------------------------------------------------------

@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("ny", EDGE_NYS)
def test_tile_width_edge_sweeps(vhp, torch, ctx, oracle, preds, ny, side):
    """Fields fp64 / fp32, bits and row runs at nx = edge (the tile kernel, bits staged as floats in rows of 301 or
    302 words) and nx = edge + 1 (grid mode for a few pairs, the naive kernel for more).  Launches of the device
    form: the tile kernel and the naive kernel 1 per batch, the bit form of the tile kernel 1, of the naive kernel
    1 + the threshold pass, grid mode 2 per pair."""
    edge = tile_edge(preds, ny)
    nx = edge + side
    assert supported(vhp, nx, ny) == (side == 0, True)
    occ, srcs, fields = edge_case(oracle, nx, ny)
    idx = np.arange(TILE_PAIRS) % len(srcs)
    xy, want = srcs[idx], fields[idx]
    what = (nx, ny)
    check_fields(vhp, ctx, occ, xy, want, what)
    check_bits_and_runs(vhp, ctx, occ, xy, want, what)

    occ_t = torch.from_numpy((occ != 0).astype(np.uint8)[None]).cuda()
    ctx.prepare_maps_dev(occ_t)
    try:
        for n, mode, want_launches in ((TILE_PAIRS, 1, 1), (len(srcs), 0 if side == 0 else 1, 1 if side == 0 else
                                                            2 * len(srcs))):
            ctx.set_grid_sweep(mode)
            xy_t = torch.from_numpy(xy[:n].copy()).cuda()
            out = torch.empty((n, ny, nx), dtype=torch.float64, device="cuda:0")
            assert launches_of(ctx, lambda: ctx.visibility_batch_dev(occ_t, xy_t, out)) == want_launches, (what, n)
            assert np.array_equal(out.cpu().numpy(), want[:n]), (what, n, mode)
            del out
        ctx.set_grid_sweep(1)
        xy_t = torch.from_numpy(xy.copy()).cuda()
        bits = torch.empty((TILE_PAIRS, ny, (nx + 31) // 32), dtype=torch.int32, device="cuda:0")
        assert launches_of(ctx, lambda: ctx.visibility_batch_bin_dev(occ_t, xy_t, THR, bits)) == 1 + side, what
        assert np.array_equal(bits.cpu().numpy().view(np.uint32), vhp.pack_bits(want >= THR)), what
    finally:
        ctx.set_grid_sweep(1)
        ctx.lib.vhp_release_maps_dev(ctx.h)


@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("ny", EDGE_NYS)
def test_tile_width_edge_merge(vhp, torch, ctx, oracle, preds, ny, side):
    """visibility_merge_batch at nx = edge (the sweep folds straight into the outputs: merge table + 1 sweep) and
    edge + 1 (the naive kernel's fp64 fields + the fold kernel), against the fold of the oracle's fields"""
    nx = tile_edge(preds, ny) + side
    occ, srcs, fields = edge_case(oracle, nx, ny)
    idx = np.arange(TILE_PAIRS) % len(srcs)
    xy, fl = srcs[idx], fields[idx]
    ptr = np.array([0, 1, 6, 11, TILE_PAIRS], np.int64)
    want = merge_expected(fl, xy, ptr, THR, (ny, nx))
    for dt in (vhp.F64, vhp.F32):
        merge_check(ctx.visibility_merge_batch(occ, xy, ptr, THR, dtype=dt), want, dt == vhp.F32, (nx, ny, dt))
    occ_t = torch.from_numpy((occ != 0).astype(np.uint8)[None]).cuda()
    xy_t = torch.from_numpy(xy.copy()).cuda()
    gptr = torch.from_numpy(ptr).cuda()
    vmax = torch.empty((len(ptr) - 1, ny, nx), dtype=torch.float64, device="cuda:0")
    ctx.prepare_maps_dev(occ_t)
    try:
        n = launches_of(ctx, lambda: ctx.visibility_merge_batch_dev(occ_t, xy_t, gptr, THR, vmax_t=vmax))
        assert n == 2 + side, (nx, ny)
        assert np.array_equal(vmax.cpu().numpy(), want[0]), (nx, ny)
    finally:
        ctx.lib.vhp_release_maps_dev(ctx.h)


@pytest.mark.parametrize("ny", EDGE_NYS)
def test_planner_width_edge(vhp, ctx, oracle, preds, ny):
    """planner_batch on the edge map with grid mode off (one persistent CTA per problem: PACK + 1 launches), and the
    same problems one column wider, where the persistent kernel is refused and the grid route runs them.  The planner's
    edge lies 32 or 64 columns below the tile kernel's (its static shared memory), so the wider map is one the tile
    kernel still sweeps; the persistent kernel failed to launch there before vhp_planner_supported counted it."""
    edge = planner_edge(preds, ny)
    max_iter = 3 if ny >= 1000 else 12
    for side in (0, 1):
        nx = edge + side
        occ = edge_case(oracle, nx, ny)[0].copy()
        se = np.array([(0, 0, nx - 1, ny - 1), (nx - 1, ny // 2, 32, 0)], np.int32)
        for x0, y0, x1, y1 in se:
            occ[y0, x0] = occ[y1, x1] = 1
        call = lambda: ctx.planner_batch(occ, se, threshold=0.25, max_iter=max_iter)  # noqa: E731
        ctx.set_grid_sweep(0)
        try:
            if side == 0:
                n, r = launches_and_result(ctx, call)
                assert n == PACK + 1, (nx, ny)
            else:
                with pytest.raises(vhp.VhpError) as e:
                    call()
                assert e.value.status == -5
                ctx.set_grid_sweep(1)
                r = call()
        finally:
            ctx.set_grid_sweep(1)
        for k, (x0, y0, x1, y1) in enumerate(se):
            planner_check(r, k, oracle.solve(occ, (x0, y0), (x1, y1), 0.25, max_iter))


# ---- the largest side ----------------------------------------------------------------------------------------------

def impl_ctx(vhp, impl):
    c = new_ctx(vhp, naive=impl == "naive")
    if impl == "grid":
        c.set_grid_sweep(2)
    return c


@pytest.mark.parametrize("impl", ["auto", "naive", "grid"])
@pytest.mark.parametrize("shape", [(MAX_SIDE, 1), (1, MAX_SIDE), (MAX_SIDE, 40), (40, MAX_SIDE)])
def test_largest_side(vhp, oracle, shape, impl):
    """maps with a side of 16384 through the automatic rule, the naive kernel and forced grid mode: fields, bits and
    row runs against the oracle"""
    nx, ny = shape
    occ, srcs, fields = edge_case(oracle, nx, ny)
    c = impl_ctx(vhp, impl)
    try:
        check_fields(vhp, c, occ, srcs, fields, (shape, impl))
        check_bits_and_runs(vhp, c, occ, srcs, fields, (shape, impl))
    finally:
        c.close()


def test_largest_square_against_the_oracle(vhp, ctx, oracle):
    """One source on a 16384 x 16384 map (nx * ny = 2^28, inside the 2^30 bound), fp64, against the oracle: grid mode,
    as the map is too wide for the one-CTA kernel.  The oracle takes about 16 s for this map on one core of an x86
    server and needs 2 GB each for its fp64 map and its field, the library's field another 2 GB; the whole map is
    compared, not a strip."""
    n = MAX_SIDE
    occ = rect_map(n, n, n * n // 4000, 5)
    sx, sy = n // 2 - 1, n // 2 - 1  # x mod 32 = 31
    got = ctx.visibility_batch(occ, [(sx, sy)], dtype=vhp.F64)[0]
    want = oracle.compute_visibility(occ, sx, sy)
    assert np.array_equal(got, want)
    assert (want > 0).sum() > n * n // 10  # the field is not trivially empty


@pytest.mark.parametrize("shape", [(MAX_SIDE + 1, 1), (1, MAX_SIDE + 1)])
def test_side_above_the_maximum_is_refused(vhp, torch, ctx, oracle, shape):
    """16385 in either dimension is VHP_ERR_UNSUPPORTED for every entry point family; the context works after"""
    nx, ny = shape
    occ = np.ones((1, ny, nx), np.uint8)
    xy, ptr = np.zeros((1, 2), np.int32), np.array([0, 1], np.int64)
    views = vhp.sensor_views(0.0, 360.0, 2)
    box = vhp.RANGE_BOX
    calls = dict(
        sweep=lambda: ctx.visibility_batch(occ, xy),
        packed=lambda: ctx.visibility_batch_packed(occ, xy),
        bits=lambda: ctx.visibility_batch_bin(occ, xy, THR),
        runs=lambda: ctx.visibility_batch_runs(occ, xy, THR),
        window=lambda: ctx.visibility_window_batch(occ, xy, 2),
        merge=lambda: ctx.visibility_merge_batch(occ, xy, ptr, THR),
        merge_range=lambda: ctx.visibility_merge_range_batch(occ, xy, ptr, THR, 2, box),
        merge_view=lambda: ctx.visibility_merge_view_batch(occ, xy, views, ptr, THR, 2, box),
        cover=lambda: ctx.visibility_cover_greedy_batch(occ, xy, ptr, 1, THR, 2, box),
        cover_weighted=lambda: ctx.visibility_cover_greedy_weighted_batch(occ, xy, ptr, 1, THR, 2, box),
        cover_mfold=lambda: ctx.visibility_cover_greedy_mfold_batch(occ, xy, ptr, 1, 2, THR, 2, box),
        cover_view=lambda: ctx.visibility_cover_greedy_view_batch(occ, xy, views, ptr, 1, 1, THR, 2, box),
        cover_quota=lambda: ctx.visibility_cover_quota_batch(occ, xy, ptr, THR, 2, box, quota=1),
        planner=lambda: ctx.planner_batch(occ, [(0, 0, 0, 0)], max_iter=2),
        raycast=lambda: ctx.raycast_batch(occ, xy),
        variant=lambda: ctx.visibility_variant_batch(occ, xy, vhp.VARIANT_QUEUE),
    )
    occ_t = torch.from_numpy(occ).cuda()
    xy_t = torch.from_numpy(xy).cuda()
    out_t = torch.empty((1, ny, nx), dtype=torch.float64, device="cuda:0")
    calls.update(sweep_dev=lambda: ctx.visibility_batch_dev(occ_t, xy_t, out_t),
                 raycast_dev=lambda: ctx.raycast_batch_dev(occ_t, xy_t, out_t))
    for name, call in calls.items():
        with pytest.raises(vhp.VhpError) as e:
            call()
        assert e.value.status == -5, name
    mx, my = min(nx, MAX_SIDE), min(ny, MAX_SIDE)
    occ_ok, srcs, fields = edge_case(oracle, mx, my)
    check_fields(vhp, ctx, occ_ok, srcs, fields, (mx, my))


# ---- the direct window route: the radius edge -------------------------------------------------------------------

def wide_sources(oracle, nx, ny):
    occ, srcs, fields = edge_case(oracle, nx, ny)
    idx = [0, 4, 5, 1, 6]  # corner, both sides of the middle tile border, the far corner, the middle
    return occ, srcs[idx], fields[idx], np.array([0, 2, 5], np.int64)


def test_window_radius_edge_wide_map(vhp, torch, ctx, oracle, preds):
    """visibility_window_batch on 16384 x 40 at R = edge (direct) and R = edge + 1 (full fields in grid mode and the
    crop), windows of 9631^2 and 9633^2 fp64, against the oracle field cropped with zeros off the grid.  The host form
    sweeps a window this large one pair per chunk, so the route is pinned on the device form: 1 launch direct, 2 grid
    kernels per pair + the crop past the edge."""
    nx, ny = MAX_SIDE, 40
    edge = window_edge(preds, nx, ny)
    occ, srcs, fields, _ = wide_sources(oracle, nx, ny)
    occ_t = torch.from_numpy((occ != 0).astype(np.uint8)[None]).cuda()
    for R, direct in ((edge, True), (edge + 1, False)):
        assert preds["window"](nx, ny, R) == direct
        for k in ((1, 3), (4,)):
            got = ctx.visibility_window_batch(occ, srcs[list(k)], R)
            for g, i in zip(got, k):
                assert np.array_equal(g, window_of(fields[i], int(srcs[i, 0]), int(srcs[i, 1]), R)), (R, i)
            xy_t = torch.from_numpy(srcs[list(k)].copy()).cuda()
            out = torch.empty((len(k), 2 * R + 1, 2 * R + 1), dtype=torch.float64, device="cuda:0")
            ctx.prepare_maps_dev(occ_t)
            try:
                n = launches_of(ctx, lambda: ctx.visibility_window_batch_dev(occ_t, xy_t, R, out))
            finally:
                ctx.lib.vhp_release_maps_dev(ctx.h)
            assert n == (1 if direct else 2 * len(k) + 1), (R, k)
            assert np.array_equal(out.cpu().numpy(), got), (R, k)
            del got, out


def test_merge_and_cover_radius_edge_wide_map(vhp, torch, ctx, oracle, preds):
    """visibility_merge_range_batch and visibility_cover_greedy_batch on 16384 x 40 at R = edge and edge + 1, box and
    disk, against their numpy references on the oracle's fields.  Range-merge launches of the device form: merge
    table + 1 sweep (direct); past the edge merge table + per 1-pair chunk of 742 MB windows the sanitised pairs,
    2 grid kernels, the crop and the fold"""
    nx, ny = MAX_SIDE, 40
    edge = window_edge(preds, nx, ny)
    occ, srcs, fields, ptr = wide_sources(oracle, nx, ny)
    occ_t = torch.from_numpy((occ != 0).astype(np.uint8)[None]).cuda()
    xy_t, gptr = torch.from_numpy(srcs.copy()).cuda(), torch.from_numpy(ptr).cuda()
    vmax = torch.empty((2, ny, nx), dtype=torch.float64, device="cuda:0")
    for R in (edge, edge + 1):
        for sh in ("box", "disk"):
            shape = vhp.RANGE_DISK if sh == "disk" else vhp.RANGE_BOX
            want = range_expected(fields, srcs, ptr, THR, (ny, nx), R, sh == "disk")
            for dt in (vhp.F64, vhp.F32):
                r = ctx.visibility_merge_range_batch(occ, srcs, ptr, THR, R, shape, dtype=dt)
                merge_check(r, want, dt == vhp.F32, (R, sh, dt))
            r = ctx.visibility_cover_greedy_batch(occ, srcs, ptr, 3, THR, R, shape)
            cover_check(vhp, r, cover_expected(fields, srcs, ptr, THR, R, sh == "disk", 3), nx, (R, sh))
        ctx.prepare_maps_dev(occ_t)
        try:
            n = launches_of(ctx, lambda: ctx.visibility_merge_range_batch_dev(occ_t, xy_t, gptr, THR, R,
                                                                               vhp.RANGE_DISK, vmax_t=vmax))
        finally:
            ctx.lib.vhp_release_maps_dev(ctx.h)
        assert n == (2 if R == edge else 1 + 5 * len(srcs)), R


def test_merge_view_radius_edge_wide_map(vhp, torch, ctx, oracle, preds):
    """visibility_merge_view_batch on 16384 x 40 at R = 4799 (direct), 4800 and 4815 (the view merge falls back while
    the range merge stays direct): omnidirectional views equal the range merge bit for bit, 90-degree views equal
    the view fold of the oracle's fields.  Launches of the device forms: merge table + 1 sweep direct; the view
    fallback merge table + per 1-pair chunk of ~740 MB windows the direct window kernel and the view fold"""
    nx, ny = MAX_SIDE, 40
    vedge, wedge = view_edge(preds, nx, ny), window_edge(preds, nx, ny)
    assert vedge < wedge
    occ, srcs, fields, ptr = wide_sources(oracle, nx, ny)
    occ_t = torch.from_numpy((occ != 0).astype(np.uint8)[None]).cuda()
    xy_t, gptr = torch.from_numpy(srcs.copy()).cuda(), torch.from_numpy(ptr).cuda()
    vmax = torch.empty((2, ny, nx), dtype=torch.float64, device="cuda:0")
    for R in (vedge, vedge + 1, wedge):
        omni = vhp.sensor_views(np.zeros(len(srcs)), 360.0, R)
        sector = vhp.sensor_views([0.0, 90.0, 180.0, 270.0, 45.0], 90.0, R)
        for sh in ("box", "disk"):
            shape = vhp.RANGE_DISK if sh == "disk" else vhp.RANGE_BOX
            want = view_expected(fields, srcs, sector, ptr, THR, R, sh)
            for dt in (vhp.F64, vhp.F32):
                rng = ctx.visibility_merge_range_batch(occ, srcs, ptr, THR, R, shape, dtype=dt)
                got = ctx.visibility_merge_view_batch(occ, srcs, omni, ptr, THR, R, shape, dtype=dt)
                for k in ("vmax", "first", "count"):
                    assert np.array_equal(got[k], rng[k]), (R, sh, dt, k)
                got = ctx.visibility_merge_view_batch(occ, srcs, sector, ptr, THR, R, shape, dtype=dt)
                merge_check(got, want, dt == vhp.F32, (R, sh, dt))
        views_t = torch.from_numpy(sector).cuda()
        ctx.prepare_maps_dev(occ_t)
        try:
            nv = launches_of(ctx, lambda: ctx.visibility_merge_view_batch_dev(occ_t, xy_t, views_t, gptr, THR, R,
                                                                              vhp.RANGE_DISK, vmax_t=vmax))
            nr = launches_of(ctx, lambda: ctx.visibility_merge_range_batch_dev(occ_t, xy_t, gptr, THR, R,
                                                                               vhp.RANGE_DISK, vmax_t=vmax))
        finally:
            ctx.lib.vhp_release_maps_dev(ctx.h)
        assert (nv, nr) == ((2, 2) if R == vedge else (1 + 2 * len(srcs), 2)), R


def test_window_radius_edge_square(vhp, torch, ctx, preds):
    """visibility_window_batch_dev on 16384 x 16384 at R = edge (direct: 1 launch) and edge + 1 (2 grid kernels per
    pair + the crop), against crops of the library's own visibility_batch_dev fields taken on the device; the
    oracle would take about 16 s per source here, and test_largest_square_against_the_oracle pins those fields"""
    n = MAX_SIDE
    edge = window_edge(preds, n, n)
    occ_t = dev_maps(torch, 1, n, n, 21)
    for xy in ([(n // 2 - 1, n // 2 - 1), (n - 1, 40)], [(4096, 12000)]):
        xy_t = torch.tensor(xy, dtype=torch.int32, device="cuda:0")
        full = torch.empty((len(xy), n, n), dtype=torch.float64, device="cuda:0")
        ctx.visibility_batch_dev(occ_t, xy_t, full)
        ctx.synchronize()
        for R, direct in ((edge, True), (edge + 1, False)):
            W = 2 * R + 1
            want = torch.zeros((len(xy), W, W), dtype=torch.float64, device="cuda:0")
            for k, (sx, sy) in enumerate(xy):
                x0, y0 = sx - R, sy - R
                xa, xb, ya, yb = max(x0, 0), min(x0 + W, n), max(y0, 0), min(y0 + W, n)
                want[k, ya - y0:yb - y0, xa - x0:xb - x0] = full[k, ya:yb, xa:xb]
            out = torch.empty_like(want)
            torch.cuda.synchronize()
            ctx.prepare_maps_dev(occ_t)
            try:
                got = launches_of(ctx, lambda: ctx.visibility_window_batch_dev(occ_t, xy_t, R, out))
            finally:
                ctx.lib.vhp_release_maps_dev(ctx.h)
            assert got == (1 if direct else 2 * len(xy) + 1), (R, xy)
            assert bool(torch.equal(out, want)), (R, xy)
            del want, out
        del full


# ---- launch-grid limits: 65 535 pairs / maps per launch ----------------------------------------------------------

RAY_CASES = [(12, 9, n) for n in (65534, 65535, 65536, 131071)] + [(1, 1, 65536), (1, 23, 65536), (23, 1, 65536)]


@pytest.mark.parametrize("nx,ny,n", RAY_CASES)
def test_raycast_pair_chunks(vhp, torch, ctx, oracle, nx, ny, n):
    """Ray casting of n pairs on two small maps with a map index per pair, host and device forms, fp64 and fp32:
    every pair against the oracle's field of its (map, source), precomputed for every cell.  Pair i casts from
    cell i mod (cells - 1 or 1) of map (i // 7) mod 2, so the pairs of the second launch differ from the first's."""
    cells = nx * ny
    occ = np.stack([rect_map(nx, ny, max(1, cells // 12), 31 + m, 1, 3) for m in range(2)])
    table = np.stack([np.stack([oracle.raycast_all(occ[m], c % nx, c // nx) for c in range(cells)])
                      for m in range(2)])  # (map, source cell, ny, nx)
    cell = np.arange(n) % max(cells - 1, 1)
    pm = ((np.arange(n) // 7) % 2).astype(np.int32)
    xy = np.stack([cell % nx, cell // nx], 1).astype(np.int32)
    want = table[pm, cell]
    for dt in (vhp.F64, vhp.F32):
        w = want if dt == vhp.F64 else f32(want)
        assert np.array_equal(ctx.raycast_batch(occ, xy, src_map=pm, dtype=dt), w), (n, dt)
        out = torch.empty((n, ny, nx), dtype=torch.float64 if dt == vhp.F64 else torch.float32, device="cuda:0")
        occ_t = torch.from_numpy((occ != 0).astype(np.uint8)).cuda()
        ctx.raycast_batch_dev(occ_t, torch.from_numpy(xy).cuda(), out, torch.from_numpy(pm).cuda())
        ctx.synchronize()
        assert np.array_equal(out.cpu().numpy(), w), (n, dt, "dev")


def test_environment_map_chunks(vhp, torch, ctx, oracle):
    """generate_environments_dev of 65 537 maps of 8 x 8: the maps on both sides of each launch's 65 535 against the
    oracle's counter-based generator, with and without a first-map offset"""
    nmaps, args = 65537, (3, 1, 4, 1, 4, 77)
    occ_t = torch.zeros((nmaps, 8, 8), dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()  # the context's stream does not wait for torch's
    for first in (0, 5):
        ctx.generate_environments_dev(occ_t, *args, first_map=first)
        ctx.synchronize()
        occ = occ_t.cpu().numpy()
        for m in (0, 1, 65534, 65535, 65536):
            want = oracle.generate_environment_counter(8, 8, *args, first + m).astype(np.uint8)
            assert np.array_equal(occ[m], want), (first, m)
        assert (occ == 0).any(axis=(1, 2)).mean() > 0.5  # obstacles in most maps
