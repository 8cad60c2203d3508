"""Directional merged visibility (vhp_visibility_merge_view_batch) on the GPU: every source alone against the numpy
definition on the direct, grid and naive routes at the 8-, 4- and 1-warp sizes, oracle parity on grouped sources,
the omnidirectional identity with vhp_visibility_merge_range_batch (also beyond the one-CTA map limit), agreement with
the view cover call, duplicate sensors, the _dev form against the host form, a host call over several runs of groups,
launch counts and every error case.  Every comparison is exact, fp64 and fp32."""
import ctypes as C

import numpy as np
import pytest

from conftest import rect_map
from test_cover_view_cpu import view_mask
from test_gpu_cover_view import contexts, seeded_views
from test_gpu_merge import THRS, check, make_groups
from test_gpu_merge_range import shape_of
from test_gpu_routes import dev_maps, host_maps, launches_of, sources
from test_merge_cpu import writes_mask
from test_merge_range_cpu import range_mask
from test_merge_view_cpu import fold_view

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


def expected(fields, srcs, views, ptr, thr, R, sh):
    outs = [fold_view(fields[ptr[g]:ptr[g + 1]], srcs[ptr[g]:ptr[g + 1]], views[ptr[g]:ptr[g + 1]], thr, R, sh)
            if ptr[g + 1] > ptr[g] else (np.zeros(fields.shape[1:]), np.full(fields.shape[1:], -1, np.int32),
                                         np.zeros(fields.shape[1:], np.uint32))
            for g in range(len(ptr) - 1)]
    return [np.stack([o[i] for o in outs]) for i in range(3)]


def omni_views(n, R):
    base = [(R, 1, 0, 1, 0), (R, 3, -7, 3, -7), (R, -32767, 5, -32767, 5), (R, 0, -1, 0, -2)]
    return np.array([base[i % len(base)] for i in range(n)], np.int32)


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the batch)
def test_every_source_alone(vhp, monkeypatch, n):
    """one group per source: vmax is the field on the view, count (and first == 0) the view's hits"""
    rng = np.random.default_rng(n + 29)
    cs = contexts(vhp, monkeypatch)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 10, 70 + m, 3, 14) for m in range(2)])
    srcs = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
    corners = [(0, 0), (nx - 1, ny - 1), (0, ny - 1), (nx - 1, 0), (31, 0), (32, ny - 1), (nx // 2, 0), (0, ny // 2),
               (63, 40), (64, 1), (nx - 2, 5)]
    srcs[:min(n, len(corners))] = corners[:n]
    gmap = rng.integers(0, 2, n).astype(np.int32)
    ptr = np.arange(n + 1, dtype=np.int64)
    fields = cs[0].visibility_batch(occ, srcs, src_map=gmap, dtype=vhp.F64)
    Y, X = np.indices((ny, nx))
    for R in (3, 20, 45):
        views = seeded_views(vhp, rng, n, R)
        for sh in SHAPES:
            masks = np.stack([range_mask(nx, ny, int(sx), int(sy), R, sh == "disk") &
                              view_mask(X - sx, Y - sy, v, R, sh) for (sx, sy), v in zip(srcs, views)])
            wr = np.stack([writes_mask(nx, ny, int(sx), int(sy)) for sx, sy in srcs])
            want_vmax = np.where(masks, fields, 0.0)
            for thr in (0.5, 0.0):  # direct route, and the fallback
                hit = masks & wr & (fields >= thr)
                for c in cs:
                    r = c.visibility_merge_view_batch(occ, srcs, views, ptr, thr, R, shape_of(vhp, sh), group_map=gmap)
                    bad = np.flatnonzero((r["count"] != hit).any((1, 2)) | (r["vmax"] != want_vmax).any((1, 2)))
                    assert not len(bad), (n, R, sh, thr, srcs[bad[0]], views[bad[0]])
                    assert np.array_equal(r["first"], np.where(hit, 0, -1).astype(np.int32)), (n, R, sh, thr)
    for c in cs:
        c.close()


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny + 31)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    sizes = [0, 1, 2, 7, 33, 0, 2]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 2 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)])
    for R in (0, 1, 31, 33, max(nx, ny) + 3):
        views = seeded_views(vhp, rng, len(srcs), R)
        for sh in SHAPES:
            for thr in THRS:  # thr <= 0: the fallback
                want = expected(fields, srcs, views, ptr, thr, R, sh)
                for dt in (vhp.F64, vhp.F32):
                    r = ctx.visibility_merge_view_batch(occ, srcs, views, ptr, thr, R, shape_of(vhp, sh),
                                                        group_map=gmap, dtype=dt)
                    check(r, want, dt == vhp.F32, (shape, R, sh, thr, dt))


def test_omni_is_the_range_merge(vhp, monkeypatch):
    """every view a == b with r = R: bit-identical to visibility_merge_range_batch on every route"""
    rng = np.random.default_rng(13)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 12, 40 + m, 3, 14) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [5, 0, 12, 1, 30])
    gmap = np.array([1, 0, 0, 1, 1], np.int32)
    cs = contexts(vhp, monkeypatch)
    for R in (0, 7, 40, 200):
        views = omni_views(len(srcs), R)
        for sh in SHAPES:
            for thr in (0.5, 1e-9, 0.0):
                for dt in (vhp.F64, vhp.F32):
                    for c in cs:
                        want = c.visibility_merge_range_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh),
                                                              group_map=gmap, dtype=dt)
                        got = c.visibility_merge_view_batch(occ, srcs, views, ptr, thr, R, shape_of(vhp, sh),
                                                            group_map=gmap, dtype=dt)
                        for k in ("vmax", "first", "count"):
                            assert np.array_equal(got[k], want[k]), (R, sh, thr, dt, k)
    for c in cs:
        c.close()


def test_omni_beyond_one_cta_map_limit(vhp):
    """12000 x 12000, R = 40: the _dev form with omnidirectional views against the range merge's _dev form"""
    import torch
    c = vhp.Context(0)
    nx = ny = 12000
    occ_t = torch.empty((1, ny, nx), dtype=torch.uint8, device="cuda:0")
    c.generate_environments_dev(occ_t, 8000, 10, 100, 10, 100, 3)
    rng = np.random.default_rng(12001)
    xy = np.concatenate([np.array([(0, 0), (11999, 11999), (31, 11999), (11968, 17), (6000, 6000), (6000, 6000)]),
                         np.stack([rng.integers(5950, 6050, 40), rng.integers(5950, 6050, 40)], 1)]).astype(np.int32)
    xy_t = torch.from_numpy(xy).cuda()
    ptr_t = torch.tensor([0, len(xy)], dtype=torch.int64, device="cuda:0")
    R = 40
    views_t = torch.from_numpy(omni_views(len(xy), R)).cuda()
    for sh in SHAPES:
        for thr in (0.5, 0.0):
            for tdt in (torch.float64, torch.float32):
                outs = []
                for view in (False, True):
                    vm = torch.full((1, ny, nx), 7.0, dtype=tdt, device="cuda:0")
                    fi = torch.full((1, ny, nx), 5, dtype=torch.int32, device="cuda:0")
                    co = torch.full((1, ny, nx), 5, dtype=torch.int32, device="cuda:0")
                    torch.cuda.synchronize()
                    if view:
                        c.visibility_merge_view_batch_dev(occ_t, xy_t, views_t, ptr_t, thr, R, shape_of(vhp, sh),
                                                          vmax_t=vm, first_t=fi, count_t=co)
                    else:
                        c.visibility_merge_range_batch_dev(occ_t, xy_t, ptr_t, thr, R, shape_of(vhp, sh), vmax_t=vm,
                                                           first_t=fi, count_t=co)
                    c.synchronize()
                    outs.append((vm, fi, co))
                for a, b in zip(*outs):
                    assert bool(torch.equal(a, b)), (sh, thr, tdt)
                assert int(outs[1][2].sum()) > 0
                del outs
    c.close()


def test_agrees_with_the_view_cover_call(ctx, vhp):
    """singletons: count == 1 exactly on S_view(c); the picks P of the view cover call: min(m, count over P) is its
    count"""
    rng = np.random.default_rng(41)
    nx, ny = 90, 70
    occ = np.stack([rect_map(nx, ny, 14, 80 + m, 3, 12) for m in range(2)])
    sizes = [9, 20, 1, 14]
    srcs, ptr = make_groups(rng, nx, ny, occ[0], sizes)
    gmap = np.array([0, 1, 1, 0], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    n = len(srcs)
    for R, sh in ((6, "disk"), (25, "box"), (40, "disk")):
        views = seeded_views(vhp, rng, n, R)
        for thr in (0.5, 0.0):
            single = ctx.visibility_cover_greedy_view_batch(occ, srcs, views, np.arange(n + 1), 1, 1, thr, R,
                                                            shape_of(vhp, sh), group_map=pmap)
            merged = ctx.visibility_merge_view_batch(occ, srcs, views, np.arange(n + 1), thr, R, shape_of(vhp, sh),
                                                     group_map=pmap, outputs=("count",))
            assert merged["count"].max() <= 1
            assert np.array_equal(merged["count"], single["count"].astype(np.uint32)), (R, sh, thr)
            for m in (1, 2, 3):
                cov = ctx.visibility_cover_greedy_view_batch(occ, srcs, views, ptr, 6, m, thr, R, shape_of(vhp, sh),
                                                             group_map=gmap)
                picks = [ptr[g] + cov["pick"][g, :cov["npicked"][g]] for g in range(len(sizes))]
                pptr = np.concatenate([[0], np.cumsum([len(p) for p in picks])]).astype(np.int64)
                idx = np.concatenate(picks).astype(np.int64)
                r = ctx.visibility_merge_view_batch(occ, srcs[idx], views[idx], pptr, thr, R, shape_of(vhp, sh),
                                                    group_map=gmap, outputs=("count",))
                assert np.array_equal(np.minimum(r["count"], m).astype(np.uint8), cov["count"]), (R, sh, thr, m)


@pytest.mark.parametrize("thr", [0.5, 0.0])  # the direct route and the fallback
def test_contention_duplicate_sensors(vhp, thr):
    """1000 sensors on one cell of an empty 1000 x 1000 map, heading four ways, and 200 more around it, one group:
    every sweep folds into the same cells at once.  Every cell in a sensor's view has value 1."""
    rng = np.random.default_rng(1000)
    n0, R = 1000, 64
    srcs = np.concatenate([np.tile([(500, 500)], (n0, 1)),
                           np.stack([rng.integers(400, 600, 200), rng.integers(400, 600, 200)], 1)]).astype(np.int32)
    c = vhp.Context(0)
    for sh in SHAPES:
        views = np.concatenate([vhp.sensor_views(np.arange(n0) % 4 * 90.0, 90, R),
                                vhp.sensor_views(rng.uniform(0, 360, 200), 120, rng.integers(0, R + 1, 200))])
        r = c.visibility_merge_view_batch(np.ones((1000, 1000)), srcs, views, [0, len(srcs)], thr, R,
                                          shape_of(vhp, sh))
        count = np.zeros((1000, 1000), np.uint32)
        first = np.full((1000, 1000), -1, np.int32)
        W = 2 * R + 1
        dy, dx = np.indices((W, W)) - R
        for k in range(len(srcs) - 1, -1, -1):
            if k < n0 and k >= 4:  # the four headings of the duplicates repeat; counted below
                continue
            sx, sy = srcs[k]
            m = view_mask(dx, dy, views[k], R, sh)
            mult = (n0 - k + 3) // 4 if k < 4 else 1
            count[sy - R:sy + R + 1, sx - R:sx + R + 1] += np.uint32(mult) * m
            first[sy - R:sy + R + 1, sx - R:sx + R + 1][m] = k
        assert np.array_equal(r["count"][0], count), sh
        assert np.array_equal(r["first"][0], first), sh
        assert np.array_equal(r["vmax"][0], (count > 0).astype(np.float64)), sh
    c.close()


def test_dev_equals_host_and_prepared_maps(vhp):
    import torch
    rng = np.random.default_rng(5)
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
        views = seeded_views(vhp, rng, len(srcs), R)
        views_t = torch.from_numpy(views).cuda()
        torch.cuda.synchronize()
        for thr in (0.5, 0.0):
            for dt, tdt in ((vhp.F64, torch.float64), (vhp.F32, torch.float32)):
                host = c.visibility_merge_view_batch(occ, srcs, views, ptr, thr, R, shape_of(vhp, sh), group_map=gmap,
                                                     dtype=dt)
                for prepared in (False, True):
                    with torch.cuda.stream(stream):
                        if prepared:
                            c.prepare_maps_dev(occ_t)
                        outs = [[torch.full((ng, ny, nx), 7.0, dtype=tdt, device="cuda:0"),
                                 torch.full((ng, ny, nx), 5, dtype=torch.int32, device="cuda:0"),
                                 torch.full((ng, ny, nx), 5, dtype=torch.int32, device="cuda:0")]
                                for _ in range(2 if prepared else 1)]
                        for vm, fi, co in outs:
                            c.visibility_merge_view_batch_dev(occ_t, xy_t, views_t, ptr_t, thr, R, shape_of(vhp, sh),
                                                              vmax_t=vm, first_t=fi, count_t=co, group_map_t=gm_t)
                    c.synchronize()
                    for vm, fi, co in outs:
                        assert np.array_equal(vm.cpu().numpy(), host["vmax"]), (R, sh, thr, dt, prepared)
                        assert np.array_equal(fi.cpu().numpy(), host["first"]), (R, sh, thr, dt, prepared)
                        assert np.array_equal(co.cpu().numpy().view(np.uint32), host["count"]), (R, sh, thr, dt)
    c.lib.vhp_release_maps_dev(c.h)
    c.close()


def test_host_call_over_several_runs_of_groups(vhp, ctx):
    """150 groups of 1000 x 1000 with all three fp64 outputs: 67 groups per 1 GB run, so three runs, each indexing
    the views at its first source; against the _dev form in one call"""
    import torch
    rng = np.random.default_rng(150)
    ng, nx, ny, R = 150, 1000, 1000, 24
    occ = host_maps(1, nx, ny, 150)
    sizes = rng.integers(0, 5, ng)
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    srcs = sources(int(ptr[-1]), nx, ny, 151)
    views = seeded_views(vhp, rng, len(srcs), R)
    host = ctx.visibility_merge_view_batch(occ, srcs, views, ptr, 0.5, R, vhp.RANGE_DISK)
    vm = torch.empty((ng, ny, nx), dtype=torch.float64, device="cuda:0")
    fi = torch.empty((ng, ny, nx), dtype=torch.int32, device="cuda:0")
    co = torch.empty((ng, ny, nx), dtype=torch.int32, device="cuda:0")
    ctx.visibility_merge_view_batch_dev(torch.from_numpy(occ).cuda(), torch.from_numpy(srcs).cuda(),
                                        torch.from_numpy(views).cuda(), torch.from_numpy(ptr).cuda(), 0.5, R,
                                        vhp.RANGE_DISK, vmax_t=vm, first_t=fi, count_t=co)
    ctx.synchronize()
    assert bool(torch.equal(vm, torch.from_numpy(host["vmax"]).cuda()))
    assert bool(torch.equal(fi, torch.from_numpy(host["first"]).cuda()))
    assert bool(torch.equal(co, torch.from_numpy(host["count"].view(np.int32)).cuda()))
    assert int(co.sum()) > 0


@pytest.mark.parametrize("mode,thr", [(1, 0.5), (1, 0.0), (2, 0.5), (2, 0.0)])
def test_launch_counts_are_the_range_merge(vhp, ctx, mode, thr):
    import torch
    nsrc, R = 5, 16
    occ_t = dev_maps(torch, 1, 1000, 1000, 7)
    xy = torch.from_numpy(sources(nsrc, 1000, 1000, 8)).cuda()
    views = torch.from_numpy(seeded_views(vhp, np.random.default_rng(8), nsrc, R)).cuda()
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    vmax = torch.empty((1, 1000, 1000), dtype=torch.float32, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        rng_call = lambda: ctx.visibility_merge_range_batch_dev(occ_t, xy, gptr, thr, R, vhp.RANGE_DISK, vmax_t=vmax)  # noqa
        view_call = lambda: ctx.visibility_merge_view_batch_dev(occ_t, xy, views, gptr, thr, R, vhp.RANGE_DISK,  # noqa
                                                                vmax_t=vmax)
        assert launches_of(ctx, view_call) == launches_of(ctx, rng_call)
    finally:
        ctx.set_grid_sweep(1)
        ctx.lib.vhp_release_maps_dev(ctx.h)


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    good = np.array([(4, 1, 0, 0, 1), (3, 1, 1, 1, 1), (0, -1, 0, 1, 0)], np.int32)
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2),
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),
        dict(group_ptr=[1, 3]),
        dict(group_ptr=[0, 2, 1, 3]),
        dict(threshold=float("nan")),
        dict(outputs=()),
    ]
    for b in bad:
        kw = dict(src_xy=srcs, views=good, group_ptr=[0, 3], threshold=0.5, radius=4, shape=vhp.RANGE_DISK)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_merge_view_batch(occ, kw.pop("src_xy"), kw.pop("views"), kw.pop("group_ptr"),
                                          kw.pop("threshold"), kw.pop("radius"), kw.pop("shape"), **kw)
        assert e.value.status == -1, b
    bad_views = [(5, 1, 0, 0, 1), (-1, 1, 0, 0, 1), (2, 0, 0, 0, 1), (2, 1, 0, 0, 0), (2, 32768, 0, 0, 1),
                 (2, 1, 0, 0, -32768)]
    for bv in bad_views:
        vw = good.copy()
        vw[1] = bv
        for s in (srcs, np.array([(1, 1), (5, 5), (70, 2)], np.int32)):  # the views are checked before the sources
            with pytest.raises(vhp.VhpError) as e:
                c.visibility_merge_view_batch(occ, s, vw, [0, 3], 0.5, 4, vhp.RANGE_DISK)
            assert e.value.status == -1
            assert b"vhp_visibility_merge_view_batch: view of source 1" in c.lib.vhp_last_error(c.h), bv
    occ_u8 = np.ones((20, 30), np.uint8)
    vp = lambda a: a.ctypes.data  # noqa: E731
    gp = np.array([0, 3], np.int64)
    cnt = np.empty((1, 20, 30), np.uint32)
    out = vhp.MergeOut(None, None, cnt.ctypes.data)
    st = c.lib.vhp_visibility_merge_view_batch(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), None, vp(gp), None, 1, 4,
                                               vhp.RANGE_BOX, 0.5, vhp.F64, C.byref(out))
    assert st == -1 and b"views is NULL" in c.lib.vhp_last_error(c.h)
    r = c.visibility_merge_view_batch(occ, srcs, good, [0, 3], 0.5, 4, vhp.RANGE_DISK)  # the context still works
    assert r["count"][0, 1, 1] == 1 and r["count"][0].max() >= 1
    # the _dev form: a bad view raises error value 16 at the next synchronising call, and its source adds nothing
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    xy_t = torch.from_numpy(srcs).to(d)
    ptr_t = torch.tensor([0, 3], dtype=torch.int64, device=d)
    for thr in (0.5, 0.0):
        for bv in bad_views:
            vw = good.copy()
            vw[1] = bv
            without = good.copy()
            without[1] = (0, 1, 0, 1, 0)  # r = 0: source 1 covers its own cell only
            want = c.visibility_merge_view_batch(occ, srcs, without, [0, 3], thr, 4, vhp.RANGE_DISK)
            want["count"][0, 5, 5] -= 1
            want["vmax"][0, 5, 5] = 0.0
            vm = torch.empty((1, 20, 30), dtype=torch.float64, device=d)
            co = torch.empty((1, 20, 30), dtype=torch.int32, device=d)
            c.visibility_merge_view_batch_dev(occ_t, xy_t, torch.from_numpy(vw).to(d), ptr_t, thr, 4, vhp.RANGE_DISK,
                                              vmax_t=vm, count_t=co)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1
            assert b"a source's view" in c.lib.vhp_last_error(c.h), (thr, bv)
            assert np.array_equal(co.cpu().numpy().view(np.uint32), want["count"]), (thr, bv)
            assert np.array_equal(vm.cpu().numpy(), want["vmax"]), (thr, bv)
        with pytest.raises(vhp.VhpError):  # NULL views at once
            c.visibility_merge_view_batch_dev(occ_t, xy_t, None, ptr_t, thr, 4, vhp.RANGE_DISK, vmax_t=vm)
    # no groups, no sources: the views are not read
    c.visibility_merge_view_batch_dev(occ_t, xy_t[:0], None, torch.zeros(1, dtype=torch.int64, device=d), 0.5, 4,
                                      vhp.RANGE_DISK, vmax_t=torch.empty((1, 20, 30), dtype=torch.float64, device=d))
    c.synchronize()
    c.close()
