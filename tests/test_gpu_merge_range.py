"""Range-limited merged visibility (vhp_visibility_merge_range_batch) on the GPU: the direct route (the sweep of each
source's box folding straight into the group outputs, 8-, 4- and 1-warp CTAs) and the fallback (fp64 windows of any
window route, folded by merge_window_fold_kernel) against the oracle, against the library's own fields and windows
(also beyond the one-CTA kernel's whole-map limit), against each other and against vhp_visibility_merge_batch.
All comparisons exact, fp64 and fp32."""
import numpy as np
import pytest

from conftest import rect_map
from test_gpu_merge import THRS, check, make_groups
from test_gpu_routes import PACK, dev_maps, launches_of, sources
from test_merge_range_cpu import fold_range

pytestmark = pytest.mark.gpu
SHAPES = ("box", "disk")


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def shape_of(vhp, name):
    return vhp.RANGE_DISK if name == "disk" else vhp.RANGE_BOX


def expected(fields, srcs, ptr, thr, shape, R, disk):
    outs = [fold_range(fields[ptr[g]:ptr[g + 1]], srcs[ptr[g]:ptr[g + 1]], thr, shape, R, disk)
            for g in range(len(ptr) - 1)]
    return [np.stack([o[i] for o in outs]) for i in range(3)]


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    sizes = [0, 1, 2, 7, 33, 0, 2]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 2 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)])
    for R in (0, 1, 31, 32, 33, max(nx, ny) + 3):
        for sh in SHAPES:
            for thr in THRS:  # thr <= 0: the fallback
                want = expected(fields, srcs, ptr, thr, (ny, nx), R, sh == "disk")
                for dt in (vhp.F64, vhp.F32):
                    r = ctx.visibility_merge_range_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), group_map=gmap,
                                                         dtype=dt)
                    check(r, want, dt == vhp.F32, (shape, R, sh, thr, dt))


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the box's size)
def test_direct_kernels_against_library_fields(vhp, n):
    rng = np.random.default_rng(n)
    c = vhp.Context(0)
    for nx, ny, nobs in ((101, 101, 10), (160, 45, 12)):
        occ = np.stack([rect_map(nx, ny, nobs, 90 + k, 3, 14) for k in range(3)])
        ngroups = 3 if n <= 12 else n // 20
        ptr = np.sort(np.concatenate([[0, n], rng.integers(0, n + 1, ngroups - 1)])).astype(np.int64)
        sizes = np.diff(ptr)
        srcs = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        srcs[:4] = [(0, 0), (nx - 1, ny - 1), (31, 5), (32 % nx, 0)]
        gmap = rng.integers(0, 3, len(sizes)).astype(np.int32)
        fields = c.visibility_batch(occ, srcs, src_map=np.repeat(gmap, sizes), dtype=vhp.F64)
        for R in (16, 40):
            for sh in SHAPES:
                for thr in (0.5, 1e-9):
                    want = expected(fields, srcs, ptr, thr, (ny, nx), R, sh == "disk")
                    for dt in (vhp.F64, vhp.F32):
                        r = c.visibility_merge_range_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), group_map=gmap,
                                                           dtype=dt)
                        check(r, want, dt == vhp.F32, (n, nx, ny, R, sh, thr, dt))
    c.close()


def torch_fold_windows(torch, win, xy, ny, nx, thr, R, disk):
    """one group's outputs folded from its fp64 windows (n, 2R+1, 2R+1) on the device, source by source"""
    d = win.device
    W = 2 * R + 1
    vmax = torch.zeros((ny, nx), dtype=torch.float64, device=d)
    first = torch.full((ny, nx), -1, dtype=torch.int32, device=d)
    count = torch.zeros((ny, nx), dtype=torch.int32, device=d)
    v, u = torch.meshgrid(torch.arange(W, device=d) - R, torch.arange(W, device=d) - R, indexing="ij")
    inr = (u * u + v * v <= R * R) if disk else torch.ones((W, W), dtype=torch.bool, device=d)
    for k, (sx, sy) in enumerate(xy.tolist()):
        x0, y0 = sx - R, sy - R
        xa, xb, ya, yb = max(x0, 0), min(x0 + W, nx), max(y0, 0), min(y0 + W, ny)
        w = win[k, ya - y0:yb - y0, xa - x0:xb - x0]
        m = inr[ya - y0:yb - y0, xa - x0:xb - x0].clone()
        vm = vmax[ya:yb, xa:xb]
        torch.maximum(vm, torch.where(m, w, torch.zeros_like(w)), out=vm)
        if sx != 0 and xa == 0:
            m[:, 0] = False  # the never-written border
        if sy != 0 and ya == 0:
            m[0, :] = False
        hit = m & (w >= thr)
        f = first[ya:yb, xa:xb]
        f[(f < 0) & hit] = k
        count[ya:yb, xa:xb] += hit.to(torch.int32)
    return vmax, first, count


def test_beyond_one_cta_map_limit(vhp):
    """12000 x 12000: too wide for the merge's direct route (whole-map state), a box of R = 40 is not.  Against
    visibility_window_batch_dev's fp64 windows folded on the device."""
    import torch
    c = vhp.Context(0)
    nx = ny = 12000
    occ_t = torch.empty((1, ny, nx), dtype=torch.uint8, device="cuda:0")
    c.generate_environments_dev(occ_t, 8000, 10, 100, 10, 100, 3)
    rng = np.random.default_rng(12000)
    xy = np.concatenate([np.array([(0, 0), (11999, 11999), (31, 11999), (11968, 17), (6000, 6000), (6000, 6000)]),
                         np.stack([rng.integers(5950, 6050, 40), rng.integers(5950, 6050, 40)], 1)]).astype(np.int32)
    xy_t = torch.from_numpy(xy).cuda()
    ptr_t = torch.tensor([0, len(xy)], dtype=torch.int64, device="cuda:0")
    R = 40
    win = torch.empty((len(xy), 2 * R + 1, 2 * R + 1), dtype=torch.float64, device="cuda:0")
    c.visibility_window_batch_dev(occ_t, xy_t, R, win)
    c.synchronize()
    for sh in SHAPES:
        for thr in (0.5, 0.0):
            want = torch_fold_windows(torch, win, xy, ny, nx, thr, R, sh == "disk")
            for tdt in (torch.float64, torch.float32):
                vm = torch.full((1, ny, nx), 7.0, dtype=tdt, device="cuda:0")
                fi = torch.full((1, ny, nx), 5, dtype=torch.int32, device="cuda:0")
                co = torch.full((1, ny, nx), 5, dtype=torch.int32, device="cuda:0")
                torch.cuda.synchronize()
                c.visibility_merge_range_batch_dev(occ_t, xy_t, ptr_t, thr, R, shape_of(vhp, sh), vmax_t=vm, first_t=fi,
                                                   count_t=co)
                c.synchronize()
                assert bool(torch.equal(vm[0], want[0].to(tdt))), (sh, thr, tdt)
                assert bool(torch.equal(fi[0], want[1])), (sh, thr, tdt)
                assert bool(torch.equal(co[0], want[2])), (sh, thr, tdt)
                del vm, fi, co
    c.close()


def test_routes_agree(vhp, monkeypatch):
    rng = np.random.default_rng(11)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 12, 40 + m, 3, 14) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [5, 0, 12, 1, 30])
    gmap = np.array([1, 0, 0, 1, 1], np.int32)
    direct = vhp.Context(0)
    grid = vhp.Context(0)
    grid.set_grid_sweep(2)
    monkeypatch.setenv("VHP_SWEEP_IMPL", "naive")
    naive = vhp.Context(0)
    monkeypatch.delenv("VHP_SWEEP_IMPL")
    for R in (0, 7, 40, 200):
        for sh in SHAPES:
            for thr in (0.5, 1e-9, 0.0):
                for dt in (vhp.F64, vhp.F32):
                    rs = [c.visibility_merge_range_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), group_map=gmap,
                                                         dtype=dt) for c in (direct, grid, naive)]
                    for r in rs[1:]:
                        for k in ("vmax", "first", "count"):
                            assert np.array_equal(r[k], rs[0][k]), (R, sh, thr, dt, k)
    for c in (direct, grid, naive):
        c.close()


def test_box_beyond_the_map_is_the_merge(vhp):
    """box with R >= max(nx, ny) - 1: bit-identical to visibility_merge_batch, on the direct route (thr > 0) and the
    fallback (thr <= 0, and grid mode forced)"""
    rng = np.random.default_rng(21)
    direct = vhp.Context(0)
    grid = vhp.Context(0)
    grid.set_grid_sweep(2)
    for nx, ny in ((101, 77), (40, 130)):
        occ = np.stack([rect_map(nx, ny, 12, 70 + m, 3, 14) for m in range(2)])
        srcs, ptr = make_groups(rng, nx, ny, occ[1], [3, 9, 0, 17])
        gmap = np.array([0, 1, 1, 0], np.int32)
        for c in (direct, grid):
            for thr in (0.5, 1e-9, 0.0, -1.0):
                for dt in (vhp.F64, vhp.F32):
                    want = c.visibility_merge_batch(occ, srcs, ptr, thr, group_map=gmap, dtype=dt)
                    for R in (max(nx, ny) - 1, max(nx, ny) + 50):
                        got = c.visibility_merge_range_batch(occ, srcs, ptr, thr, R, vhp.RANGE_BOX, group_map=gmap,
                                                             dtype=dt)
                        for k in ("vmax", "first", "count"):
                            assert np.array_equal(got[k], want[k]), (nx, ny, thr, dt, R, k)
    direct.close()
    grid.close()


def test_dev_equals_host_and_prepared_maps(vhp):
    import torch
    rng = np.random.default_rng(3)
    nx, ny = 130, 96
    occ = np.stack([rect_map(nx, ny, 15, 60 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    srcs, ptr = make_groups(rng, nx, ny, occ[2], [4, 9, 0, 1, 40, 3])
    gmap = np.array([2, 0, 1, 2, 1, 0], np.int32)
    stream = torch.cuda.Stream()
    c = vhp.torch_context(0, stream)
    occ_t, xy_t, ptr_t, gm_t = (torch.from_numpy(a).cuda() for a in (occ, srcs, ptr, gmap))
    torch.cuda.synchronize()
    ng = len(ptr) - 1
    for R, sh in ((5, "disk"), (33, "box"), (60, "disk")):
        for thr in (0.5, 0.0):
            for dt, tdt in ((vhp.F64, torch.float64), (vhp.F32, torch.float32)):
                host = c.visibility_merge_range_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), group_map=gmap,
                                                      dtype=dt)
                for prepared in (False, True):
                    with torch.cuda.stream(stream):
                        if prepared:
                            c.prepare_maps_dev(occ_t)  # the packed planes of vhp_prepare_maps_dev, used twice
                        outs = [[torch.full((ng, ny, nx), 7.0, dtype=tdt, device="cuda:0"),
                                 torch.full((ng, ny, nx), 5, dtype=torch.int32, device="cuda:0"),
                                 torch.full((ng, ny, nx), 5, dtype=torch.int32, device="cuda:0")]
                                for _ in range(2 if prepared else 1)]
                        for vm, fi, co in outs:
                            c.visibility_merge_range_batch_dev(occ_t, xy_t, ptr_t, thr, R, shape_of(vhp, sh), vmax_t=vm,
                                                               first_t=fi, count_t=co, group_map_t=gm_t)
                    c.synchronize()
                    for vm, fi, co in outs:
                        assert np.array_equal(vm.cpu().numpy(), host["vmax"]), (R, sh, thr, dt, prepared)
                        assert np.array_equal(fi.cpu().numpy(), host["first"]), (R, sh, thr, dt, prepared)
                        assert np.array_equal(co.cpu().numpy().view(np.uint32), host["count"]), (R, sh, thr, dt)
    c.lib.vhp_release_maps_dev(c.h)
    c.close()


@pytest.mark.parametrize("thr", [0.5, 0.0])  # the direct route and the fallback
def test_contention_duplicate_sensors(vhp, thr):
    """3000 sensors on one cell of an empty 1000 x 1000 map and 500 more around it, one group: every sweep folds
    into the same cells at once.  Every cell in range of a sensor has value 1."""
    rng = np.random.default_rng(3000)
    n0, R = 3000, 64
    srcs = np.concatenate([np.tile([(500, 500)], (n0, 1)),
                           np.stack([rng.integers(400, 600, 500), rng.integers(400, 600, 500)], 1)]).astype(np.int32)
    ys, xs = np.mgrid[0:1000, 0:1000]
    c = vhp.Context(0)
    for sh in SHAPES:
        r = c.visibility_merge_range_batch(np.ones((1000, 1000)), srcs, [0, len(srcs)], thr, R, shape_of(vhp, sh))
        count = np.zeros((1000, 1000), np.uint32)
        first = np.full((1000, 1000), -1, np.int32)
        for k in range(len(srcs) - 1, n0 - 1, -1):
            sx, sy = srcs[k]
            m = ((xs - sx) ** 2 + (ys - sy) ** 2 <= R * R) if sh == "disk" else (
                (abs(xs - sx) <= R) & (abs(ys - sy) <= R))
            count += m
            first[m] = k
        m0 = ((xs - 500) ** 2 + (ys - 500) ** 2 <= R * R) if sh == "disk" else (
            (abs(xs - 500) <= R) & (abs(ys - 500) <= R))
        count += np.uint32(n0) * m0
        first[m0] = 0
        assert np.array_equal(r["count"][0], count), sh
        assert np.array_equal(r["first"][0], first), sh
        assert np.array_equal(r["vmax"][0], (count > 0).astype(np.float64)), sh
    c.close()


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2), dict(shape=-1),
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),  # source outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                    # map out of range
        dict(group_ptr=[1, 3]),                                         # does not start at 0
        dict(group_ptr=[0, 2, 1, 3]),                                   # decreasing
        dict(threshold=float("nan")),
        dict(outputs=()),
    ]
    for b in bad:
        kw = dict(src_xy=srcs, group_ptr=[0, 3], threshold=0.5, radius=4, shape=vhp.RANGE_DISK)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_merge_range_batch(occ, kw.pop("src_xy"), kw.pop("group_ptr"), kw.pop("threshold"),
                                           kw.pop("radius"), kw.pop("shape"), **kw)
        assert e.value.status == -1, b
        r = c.visibility_merge_range_batch(occ, srcs, [0, 3], 0.5, 4, vhp.RANGE_DISK)  # the context still works
        assert r["count"][0].max() == 3  # e.g. (4, 2) is in range of all three
    # the _dev form: bad arguments at once, a bad source / group layout through the device error flag
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    vm = torch.empty((2, 20, 30), dtype=torch.float64, device=d)
    xy_ok = torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d)
    ptr_ok = torch.tensor([0, 1, 3], dtype=torch.int64, device=d)
    for radius, shape in ((-1, vhp.RANGE_BOX), (16384, vhp.RANGE_BOX), (4, 2)):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_merge_range_batch_dev(occ_t, xy_ok, ptr_ok, 0.5, radius, shape, vmax_t=vm)
        assert e.value.status == -1
    for thr in (0.5, 0.0):
        for xy, ptr in (([(1, 1), (31, 1), (2, 2)], [0, 1, 3]), ([(1, 1), (3, 1), (2, 2)], [0, 2, 1])):
            c.visibility_merge_range_batch_dev(occ_t, torch.tensor(xy, dtype=torch.int32, device=d),
                                               torch.tensor(ptr, dtype=torch.int64, device=d), thr, 4, vhp.RANGE_BOX,
                                               vmax_t=vm)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1, (thr, xy, ptr)
    c.visibility_merge_range_batch_dev(occ_t, xy_ok, ptr_ok, 0.5, 4, vhp.RANGE_BOX, vmax_t=vm)
    c.synchronize()
    assert (vm[0] == 1.0).sum().item() == 25  # the box of (1, 1) on the grid, without column 0 and row 0
    c.close()


@pytest.mark.parametrize("mode,thr,want", [(1, 0.5, 2), (1, 0.0, 3), (2, 0.5, 14), (2, 0.0, 14)])
def test_routes_by_launch_count(vhp, ctx, mode, thr, want):
    """direct: merge table + one sweep; fallback: merge table + per chunk the window route (the windowed kernel, or
    with grid mode forced: sanitised pairs + 2 grid kernels per pair + crop) + the window fold"""
    import torch
    nsrc, R = 5, 16
    occ_t = dev_maps(torch, 1, 1000, 1000, 7)
    xy = torch.from_numpy(sources(nsrc, 1000, 1000, 8)).cuda()
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    vmax = torch.empty((1, 1000, 1000), dtype=torch.float32, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        call = lambda: ctx.visibility_merge_range_batch_dev(occ_t, xy, gptr, thr, R, vhp.RANGE_DISK, vmax_t=vmax)  # noqa
        assert launches_of(ctx, call) == want
    finally:
        ctx.set_grid_sweep(1)


def test_host_form_packs_once(vhp, ctx):
    import test_gpu_routes
    occ = test_gpu_routes.host_maps(1, 1000, 1000, 11)
    xy = sources(5, 1000, 1000, 12)
    assert launches_of(ctx, lambda: ctx.visibility_merge_range_batch(occ, xy, [0, 5], 0.5, 16, vhp.RANGE_BOX)) == PACK + 2
    assert launches_of(ctx, lambda: ctx.visibility_merge_range_batch(occ, xy, [0, 5], 0.0, 16, vhp.RANGE_BOX)) == PACK + 3
