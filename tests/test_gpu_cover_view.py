"""Directional greedy sensor placement (vhp_visibility_cover_greedy_view_batch) on the GPU: every candidate's masked
coverage set against view_mask of test_cover_view_cpu, the full greedy against the numpy m-fold greedy on the oracle's
fields, the omnidirectional identity with vhp_visibility_cover_greedy_mfold_batch, the _dev form against the host form,
a host call over two 4 GB batches, launch counts and every error case.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

from conftest import rect_map
from test_cover_cpu import cover_set
from test_cover_view_cpu import view_mask, view_sets
from test_cover_weighted_cpu import seeded_weights
from test_gpu_cover_mfold import check, mgreedy_all
from test_gpu_cover_weighted import problem_sets, shape_of
from test_gpu_merge import make_groups
from test_gpu_routes import dev_maps, launches_of, sources

pytestmark = pytest.mark.gpu
SHAPES = ("box", "disk")

# sector edges: axis-aligned, +-32767 components, non-primitive (2, 4) with (1, 2), and a sub-degree pair
SPECIAL = [((1, 0), (0, 1)), ((0, 1), (-1, 0)), ((32767, 0), (0, -32767)), ((-32767, 32767), (32767, 32767)),
           ((2, 4), (1, 2)), ((1, 2), (2, 4)), ((32767, 100), (32767, 101)), ((32767, 101), (32767, 100)),
           ((0, -1), (0, -1)), ((-32767, -32767), (32767, 32767)), ((3, -7), (-3, 7)), ((1, 0), (-1, -1)),
           ((-1, 0), (-32767, 1)), ((-32767, 1), (-32767, -1)), ((5, 5), (5, -5))]


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def seeded_views(vhp, rng, n, R):
    """n views: the SPECIAL pairs, sensor_views sectors (90, 180, 270, 359.9, 360 degrees and 0.5 degrees) and random
    integer vectors, with r from 0 to R"""
    out = []
    for i in range(n):
        kind = i % 3
        if kind == 0:
            a, b = SPECIAL[(i // 3) % len(SPECIAL)]
            v = [0, *a, *b]
        elif kind == 1:
            fov = (90, 180, 270, 359.9, 360, 0.5, 45)[(i // 3) % 7]
            v = vhp.sensor_views(float(rng.uniform(0, 360)), fov, 0)[0].tolist()
        else:
            a = [int(t) for t in rng.integers(-32767, 32768, 2)]
            b = [int(t) for t in rng.integers(-40, 41, 2)]
            if rng.random() < 0.5:
                a, b = b, a
            a = a if a != [0, 0] else [0, 1]
            b = b if b != [0, 0] else [1, 0]
            v = [0, *a, *b]
        v[0] = R if i % 7 == 0 else 0 if i % 11 == 0 else int(rng.integers(0, R + 1))
        out.append(v)
    return np.array(out, np.int32)


def contexts(vhp, monkeypatch):
    direct = vhp.Context(0)
    grid = vhp.Context(0)
    grid.set_grid_sweep(2)
    monkeypatch.setenv("VHP_SWEEP_IMPL", "naive")
    naive = vhp.Context(0)
    monkeypatch.delenv("VHP_SWEEP_IMPL")
    return direct, grid, naive


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the batch)
def test_mask_is_exact(vhp, monkeypatch, n):
    """one problem per candidate, k = 1, weights 1: count is S_view(c), or all zero when it is empty"""
    rng = np.random.default_rng(n + 17)
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
            for thr in (0.5, 0.0):  # direct route, and the fallback
                want = np.stack([cover_set(f, int(sx), int(sy), thr, R, sh == "disk") &
                                 view_mask(X - sx, Y - sy, v, R, sh) for f, (sx, sy), v in zip(fields, srcs, views)])
                for c in cs:
                    r = c.visibility_cover_greedy_view_batch(occ, srcs, views, ptr, 1, 1, thr, R, shape_of(vhp, sh),
                                                             group_map=gmap)
                    got = r["count"].astype(bool)
                    bad = np.flatnonzero((got != want).any((1, 2)))
                    assert not len(bad), (n, R, sh, thr, srcs[bad[0]], views[bad[0]])
                    assert np.array_equal(r["npicked"], want.any((1, 2)).astype(np.int32))
                    assert np.array_equal(r["gain"][:, 0], want.sum((1, 2)).astype(np.uint64))
    for c in cs:
        c.close()


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny + 9)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    sizes = [0, 1, 2, 7, 33, 0, 2]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 2 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)])
    weights = seeded_weights((len(sizes), ny, nx), rng)
    ks = (1, 4, 8)
    for R in (0, 1, 32, max(nx, ny) + 3):
        views = seeded_views(vhp, rng, len(srcs), R)
        for sh in SHAPES:
            for thr in (0.5, 0.0):
                psets = problem_sets(fields, srcs, ptr, thr, R, sh == "disk")
                psets = [view_sets(s, srcs[a:b], views[a:b], R, sh) for s, a, b in zip(psets, ptr[:-1], ptr[1:])]
                for m in (1, 2, 3):
                    for w in (weights, None):
                        want = mgreedy_all(psets, ks, m, (ny, nx), w)
                        for k in ks:
                            r = ctx.visibility_cover_greedy_view_batch(occ, srcs, views, ptr, k, m, thr, R,
                                                                       shape_of(vhp, sh), weights=w, group_map=gmap)
                            check(r, want[k], (shape, R, sh, thr, m, k, w is None))


def omni(n, R, rng):
    a = rng.integers(-32767, 32768, (n, 2))
    a[(a == 0).all(1)] = (1, 0)
    return np.concatenate([np.full((n, 1), R), a, a], 1).astype(np.int32)


def test_omnidirectional_views_are_the_mfold_call(ctx, vhp):
    rng = np.random.default_rng(23)
    nx, ny = 150, 110
    occ = np.stack([rect_map(nx, ny, 30, 50 + m, 3, 16) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [50, 0, 1, 120, 9])
    gmap = np.array([0, 1, 0, 1, 1], np.int32)
    W = seeded_weights((len(ptr) - 1, ny, nx), rng)
    for R, sh, thr, k, m in ((20, "disk", 0.5, 9, 1), (70, "box", 1e-9, 6, 2), (12, "box", 0.0, 12, 3),
                             (200, "disk", -1.0, 3, 2), (33, "disk", 0.0, 7, 1)):
        for w in (W, None):
            u = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, k, m, thr, R, shape_of(vhp, sh), weights=w,
                                                        group_map=gmap)
            r = ctx.visibility_cover_greedy_view_batch(occ, srcs, omni(len(srcs), R, rng), ptr, k, m, thr, R,
                                                       shape_of(vhp, sh), weights=w, group_map=gmap)
            for key in ("pick", "gain", "npicked", "count"):
                assert np.array_equal(r[key], u[key]), (R, sh, thr, w is None, key)


def test_omnidirectional_identity_on_a_12000_map(vhp):
    import torch
    c = vhp.Context(0)
    nx = ny = 12000
    occ_t = torch.empty((1, ny, nx), dtype=torch.uint8, device="cuda:0")
    c.generate_environments_dev(occ_t, 8000, 10, 100, 10, 100, 5)
    rng = np.random.default_rng(12003)
    xy = np.concatenate([np.array([(0, 0), (11999, 11999), (31, 11999), (11968, 17), (6000, 6000)]),
                         np.stack([rng.integers(5800, 6200, 59), rng.integers(5800, 6200, 59)], 1)]).astype(np.int32)
    occ = occ_t.cpu().numpy()
    ptr = np.array([0, len(xy)], np.int64)
    W = rng.integers(0, 256, (1, ny, nx), dtype=np.uint8)
    for R, sh, thr in ((64, "disk", 0.5), (40, "box", 0.0)):
        u = c.visibility_cover_greedy_mfold_batch(occ, xy, ptr, 8, 2, thr, R, shape_of(vhp, sh), weights=W)
        r = c.visibility_cover_greedy_view_batch(occ, xy, omni(len(xy), R, rng), ptr, 8, 2, thr, R, shape_of(vhp, sh),
                                                 weights=W)
        for key in ("pick", "gain", "npicked", "count"):
            assert np.array_equal(r[key], u[key]), (R, sh, key)
        assert r["npicked"][0] == 8
    c.close()


def test_dev_equals_host(vhp):
    import torch
    rng = np.random.default_rng(8)
    nx, ny = 130, 96
    occ = np.stack([rect_map(nx, ny, 15, 60 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    srcs, ptr = make_groups(rng, nx, ny, occ[2], [4, 9, 0, 1, 40, 3])
    gmap = np.array([2, 0, 1, 2, 1, 0], np.int32)
    ng = len(ptr) - 1
    W = seeded_weights((ng, ny, nx), rng)
    stream = torch.cuda.Stream()
    c = vhp.torch_context(0, stream)
    occ_t, xy_t, ptr_t, gm_t, w_t = (torch.from_numpy(a).cuda() for a in (occ, srcs, ptr, gmap, W))
    torch.cuda.synchronize()
    for R, sh, thr, k, m in ((5, "disk", 0.5, 7, 2), (33, "box", 0.0, 3, 3), (60, "disk", 1e-9, 50, 1)):
        views = seeded_views(vhp, rng, len(srcs), R)
        v_t = torch.from_numpy(views).cuda()
        for w in (None, W):
            host = c.visibility_cover_greedy_view_batch(occ, srcs, views, ptr, k, m, thr, R, shape_of(vhp, sh),
                                                        weights=w, group_map=gmap)
            with torch.cuda.stream(stream):
                pk = torch.full((ng, k), 5, dtype=torch.int32, device="cuda:0")
                gn = torch.full((ng, k), 5, dtype=torch.int64, device="cuda:0")
                npk = torch.full((ng,), 5, dtype=torch.int32, device="cuda:0")
                cnt = torch.full((ng, ny, nx), 5, dtype=torch.uint8, device="cuda:0")
                c.visibility_cover_greedy_view_batch_dev(occ_t, xy_t, v_t, ptr_t, k, m, thr, R, shape_of(vhp, sh),
                                                         pick_t=pk, gain_t=gn, npicked_t=npk, count_t=cnt,
                                                         group_map_t=gm_t, weights_t=None if w is None else w_t)
            c.synchronize()
            assert np.array_equal(pk.cpu().numpy(), host["pick"]), (R, sh, thr)
            assert np.array_equal(gn.cpu().numpy().view(np.uint64), host["gain"]), (R, sh, thr)
            assert np.array_equal(npk.cpu().numpy(), host["npicked"]), (R, sh, thr)
            assert np.array_equal(cnt.cpu().numpy(), host["count"]), (R, sh, thr)
    c.close()


def test_two_4gb_batches_equal_one_problem_at_a_time(ctx, vhp):
    """8 weighted problems on 12000^2 maps with count: about 0.6 GB of device memory each, so the host form runs them
    in two batches"""
    nx = ny = 12000
    rng = np.random.default_rng(41)
    occ = np.stack([rect_map(nx, ny, 3000, 200 + m, 10, 80) for m in range(2)]).astype(np.uint8)
    sizes = [5, 1, 9, 3, 6, 2, 7, 4]
    xy = np.stack([rng.integers(0, nx, sum(sizes)), rng.integers(0, ny, sum(sizes))], 1).astype(np.int32)
    xy[:3] = [(0, 0), (nx - 1, ny - 1), (6000, 0)]
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    gmap = (np.arange(8) % 2).astype(np.int32)
    W = rng.integers(0, 256, (8, ny, nx), dtype=np.uint8)
    R = 48
    views = seeded_views(vhp, rng, len(xy), R)
    r = ctx.visibility_cover_greedy_view_batch(occ, xy, views, ptr, 4, 2, 0.5, R, vhp.RANGE_DISK, weights=W,
                                               group_map=gmap)
    for q in range(8):
        a, b = ptr[q], ptr[q + 1]
        one = ctx.visibility_cover_greedy_view_batch(occ, xy[a:b], views[a:b], [0, b - a], 4, 2, 0.5, R,
                                                     vhp.RANGE_DISK, weights=W[q:q + 1], group_map=gmap[q:q + 1])
        for key in ("pick", "gain", "npicked", "count"):
            assert np.array_equal(r[key][q], one[key][0]), (q, key)
    assert (r["npicked"] > 0).all()


@pytest.mark.parametrize("mode,thr,k,count", [(1, 0.5, 3, True), (1, 0.5, 3, False), (1, 0.5, 10, True),
                                              (1, 0.0, 3, True), (1, 0.0, 3, False), (2, 0.5, 3, True)])
def test_launches_are_the_mfold_calls_plus_one(vhp, ctx, mode, thr, k, count):
    import torch
    nsrc, R = 5, 16
    occ_t = dev_maps(torch, 1, 1000, 1000, 7)
    xy = torch.from_numpy(sources(nsrc, 1000, 1000, 8)).cuda()
    views = torch.from_numpy(vhp.sensor_views(np.arange(nsrc) * 70.0, 90, R)).cuda()
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    pk = torch.empty((1, max(k, 1)), dtype=torch.int32, device="cuda:0")
    cnt = torch.empty((1, 1000, 1000), dtype=torch.uint8, device="cuda:0") if count else None
    w = torch.ones((1, 1000, 1000), dtype=torch.uint8, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        mf = lambda: ctx.visibility_cover_greedy_mfold_batch_dev(occ_t, xy, gptr, k, 2, thr, R,  # noqa: E731
                                                                 vhp.RANGE_DISK, pick_t=pk, count_t=cnt, weights_t=w)
        vw = lambda: ctx.visibility_cover_greedy_view_batch_dev(occ_t, xy, views, gptr, k, 2, thr, R,  # noqa: E731
                                                                vhp.RANGE_DISK, pick_t=pk, count_t=cnt, weights_t=w)
        assert launches_of(ctx, vw) == launches_of(ctx, mf) + 1
    finally:
        ctx.set_grid_sweep(1)


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    good = np.array([(4, 1, 0, 0, 1), (4, 1, 1, 1, 1), (0, -1, 0, 1, 0)], np.int32)
    bad_views = [(-1, 1, 0, 0, 1), (5, 1, 0, 0, 1), (4, 0, 0, 0, 1), (4, 1, 0, 0, 0), (4, 32768, 0, 0, 1),
                 (4, 1, -32768, 0, 1), (4, 1, 0, 32768, 1), (4, 1, 0, 0, -32768)]
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2), dict(shape=-1), dict(k=-1), dict(m=0), dict(m=256),
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),  # candidate outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                 # map out of range
        dict(group_ptr=[1, 3]),                                      # does not start at 0
        dict(group_ptr=[0, 2, 1, 3]),                                # decreasing
        dict(threshold=float("nan")),
    ] + [dict(views=np.array([good[0], v, good[2]], np.int32)) for v in bad_views]
    for b in bad:
        kw = dict(src_xy=srcs, views=good, group_ptr=[0, 3], k=2, m=2, threshold=0.5, radius=4, shape=vhp.RANGE_DISK)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_view_batch(occ, kw.pop("src_xy"), kw.pop("views"), kw.pop("group_ptr"),
                                                 kw.pop("k"), kw.pop("m"), kw.pop("threshold"), kw.pop("radius"),
                                                 kw.pop("shape"), **kw)
        assert e.value.status == -1, b
        if "views" in b:
            assert b"view of candidate 1" in c.lib.vhp_last_error(c.h), b
        r = c.visibility_cover_greedy_view_batch(occ, srcs, good, [0, 3], 2, 2, 0.5, 4, vhp.RANGE_DISK)  # still works
        assert r["npicked"][0] == 2
    occ_u8 = np.ones((1, 20, 30), np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    npk = np.zeros(1, np.int32)
    one = vhp.CoverMfoldOut(None, None, npk.ctypes.data, None)
    gp = np.array([0, 3], np.int64)
    fn = c.lib.vhp_visibility_cover_greedy_view_batch
    st = fn(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), None, vp(gp), None, 1, 2, 4, vhp.RANGE_BOX, 0.5, None, 2,
            C.byref(one))
    assert st == -1 and b"views is NULL" in c.lib.vhp_last_error(c.h)
    none = vhp.CoverMfoldOut(None, None, None, None)
    st = fn(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), vp(good), vp(gp), None, 1, 2, 4, vhp.RANGE_BOX, 0.5, None, 2,
            C.byref(none))
    assert st == -1 and b"no output" in c.lib.vhp_last_error(c.h)
    big = np.array([0, 2**28], np.int64)
    st = fn(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), vp(good), vp(big), None, 1, 2, 4, vhp.RANGE_BOX, 0.5, None, 2,
            C.byref(one))
    assert st == -1 and b"2^28" in c.lib.vhp_last_error(c.h)
    # the views are checked before any candidate is read: a bad view wins over a candidate outside the grid
    st = fn(c.h, vp(occ_u8), 1, 30, 20, vp(np.array([(1, 1), (30, 5), (7, 2)], np.int32)),
            vp(np.array([good[0], good[1], (9, 1, 0, 0, 1)], np.int32)), vp(gp), None, 1, 2, 4, vhp.RANGE_BOX, 0.5,
            None, 2, C.byref(one))
    assert st == -1 and b"view of candidate 2" in c.lib.vhp_last_error(c.h)
    r = c.visibility_cover_greedy_view_batch(occ, srcs, good, [0, 3], 0, 2, 0.5, 4, vhp.RANGE_DISK)  # k = 0 is valid
    assert r["pick"].shape == (1, 0) and r["npicked"][0] == 0 and not r["count"].any()
    # the _dev form: bad arguments at once, a bad view / candidate / group layout through the device error flag
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    pk = torch.empty((2, 3), dtype=torch.int32, device=d)
    xy_ok = torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d)
    v_ok = torch.from_numpy(good).cuda()
    ptr_ok = torch.tensor([0, 1, 3], dtype=torch.int64, device=d)
    for radius, shape, k, m, thr in ((-1, vhp.RANGE_BOX, 3, 2, 0.5), (16384, vhp.RANGE_BOX, 3, 2, 0.5),
                                     (4, 2, 3, 2, 0.5), (4, vhp.RANGE_BOX, -1, 2, 0.5),
                                     (4, vhp.RANGE_BOX, 3, 2, float("nan")), (4, vhp.RANGE_BOX, 3, 0, 0.5)):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_view_batch_dev(occ_t, xy_ok, v_ok, ptr_ok, k, m, thr, radius, shape, pick_t=pk)
        assert e.value.status == -1
    c.synchronize()
    before = c.launches
    with pytest.raises(vhp.VhpError) as e:
        c.visibility_cover_greedy_view_batch_dev(occ_t, xy_ok, None, ptr_ok, 3, 2, 0.5, 4, vhp.RANGE_BOX, pick_t=pk)
    assert e.value.status == -1 and b"views is NULL" in c.lib.vhp_last_error(c.h) and c.launches == before
    for thr in (0.5, 0.0):
        for v in bad_views:
            views = torch.tensor([good[0].tolist(), list(v), good[2].tolist()], dtype=torch.int32, device=d)
            c.visibility_cover_greedy_view_batch_dev(occ_t, xy_ok, views, ptr_ok, 3, 2, thr, 4, vhp.RANGE_BOX,
                                                     pick_t=pk)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1 and b"view" in c.lib.vhp_last_error(c.h), (thr, v)
            # the bad view's candidate covers nothing; the next call on the context succeeds
            c.visibility_cover_greedy_view_batch_dev(occ_t, xy_ok, v_ok, ptr_ok, 3, 2, thr, 4, vhp.RANGE_BOX,
                                                     pick_t=pk)
            c.synchronize()
        for xy, ptr in (([(1, 1), (31, 1), (2, 2)], [0, 1, 3]), ([(1, 1), (3, 1), (2, 2)], [0, 2, 1])):
            c.visibility_cover_greedy_view_batch_dev(occ_t, torch.tensor(xy, dtype=torch.int32, device=d), v_ok,
                                                     torch.tensor(ptr, dtype=torch.int64, device=d), 3, 2, thr, 4,
                                                     vhp.RANGE_BOX, pick_t=pk)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1 and b"view" not in c.lib.vhp_last_error(c.h), (thr, xy, ptr)
    # a bad view covers nothing: problem 1 = candidates 1 (bad) and 2, so only 2 is picked
    views = torch.tensor([good[0].tolist(), [9, 1, 0, 0, 1], good[2].tolist()], dtype=torch.int32, device=d)
    gn = torch.empty((2, 3), dtype=torch.int64, device=d)
    c.visibility_cover_greedy_view_batch_dev(occ_t, xy_ok, views, ptr_ok, 3, 2, 0.5, 4, vhp.RANGE_BOX, pick_t=pk,
                                             gain_t=gn)
    with pytest.raises(vhp.VhpError):
        c.synchronize()
    assert pk[1].tolist() == [1, -1, -1]
    c.visibility_cover_greedy_view_batch_dev(occ_t, xy_ok, v_ok, ptr_ok, 3, 2, 0.5, 4, vhp.RANGE_BOX, pick_t=pk,
                                             gain_t=gn)
    c.synchronize()
    # problem 0: (1, 1) with the quarter dx >= 0, dy >= 0 (a = (1, 0), b = (0, 1)) and r = 4: 25 cells; problem 1:
    # (3, 1) sees all of its box, 7 x 5 written cells, then (2, 2), whose view of r = 0 is its own cell
    assert pk.tolist() == [[0, -1, -1], [0, 1, -1]]
    assert gn.tolist() == [[25, 0, 0], [35, 1, 0]]
    c.close()
