"""Quota sensor placement (vhp_visibility_cover_quota_batch) on the GPU: the prefix identity with the view call (views
given) or the m-fold call (views NULL) on every route and warp size, problems stopping for different reasons in one
call, a loop of thousands of rounds, kmax, launch counts, graph freshness across calls that grow the buffers, the _dev
form against the host form, a host call over two 4 GB runs, and every error case.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

from conftest import rect_map
from test_cover_weighted_cpu import seeded_weights
from test_gpu_cover_view import contexts, seeded_views
from test_gpu_cover_weighted import shape_of
from test_gpu_merge import make_groups
from test_gpu_routes import dev_maps, launches_of, sources

pytestmark = pytest.mark.gpu
U64_MAX = np.iinfo(np.uint64).max


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def reference(c, occ, srcs, views, ptr, k, m, thr, R, shape, weights, gmap):
    """the view call (views given) or the m-fold call (views None) with k picks"""
    if views is None:
        return c.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, k, m, thr, R, shape, weights=weights,
                                                     group_map=gmap)
    return c.visibility_cover_greedy_view_batch(occ, srcs, views, ptr, k, m, thr, R, shape, weights=weights,
                                                group_map=gmap)


def prefix_npicked(gain, n, quota):
    """min { j : sum of gain[:j] >= quota }, limited by n (gain 0) -- the prefix rule"""
    s = 0
    for j in range(n + 1):
        if s >= quota:
            return j
        if j < n:
            s += int(gain[j])
    return n


def check_prefix(c, occ, srcs, views, ptr, kmax, m, thr, R, shape, weights, gmap, quota, r, what):
    """r (the quota call) against the reference with k = kmax (pick, gain, npicked, total) and with k = npicked
    (count)"""
    full = reference(c, occ, srcs, views, ptr, kmax, m, thr, R, shape, weights, gmap)
    want_n = np.array([prefix_npicked(full["gain"][q], int(full["npicked"][q]), int(quota[q]))
                       for q in range(len(quota))], np.int32)
    assert np.array_equal(r["npicked"], want_n), (what, r["npicked"], want_n)
    for q, j in enumerate(want_n):
        pick, gain = full["pick"][q].copy(), full["gain"][q].copy()
        pick[j:], gain[j:] = -1, 0
        assert np.array_equal(r["pick"][q], pick), (what, q)
        assert np.array_equal(r["gain"][q], gain), (what, q)
        assert int(r["total"][q]) == int(gain.sum(dtype=np.uint64)), (what, q)
        assert bool(r["reached"][q]) == (int(r["total"][q]) >= int(quota[q])), (what, q)
    for j in np.unique(want_n):
        cut = reference(c, occ, srcs, views, ptr, int(j), m, thr, R, shape, weights, gmap)
        for q in np.flatnonzero(want_n == j):
            assert np.array_equal(r["count"][q], cut["count"][q]), (what, q, j)


def quotas_for(full, rng):
    """per problem: 0, 1, an exact prefix sum, a prefix sum + 1, unreachable, UINT64_MAX, in turn"""
    out = []
    for q in range(len(full["npicked"])):
        n = int(full["npicked"][q])
        sums = np.cumsum(full["gain"][q][:n].astype(np.int64))
        tot = int(sums[-1]) if n else 0
        j = int(rng.integers(0, n)) if n else 0
        out.append([0, 1, int(sums[j]) if n else 0, int(sums[j]) + 1 if n else 1, tot + 1, U64_MAX][q % 6])
    return np.array(out, np.uint64)


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the batch)
def test_prefix_identity(vhp, monkeypatch, n):
    rng = np.random.default_rng(n + 101)
    cs = contexts(vhp, monkeypatch)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 10, 70 + m, 3, 14) for m in range(2)])
    sizes = [0, 1, 2, 3, 6] if n == 12 else [n // 3, 1, n // 3, 0, n - 2 * (n // 3) - 1]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = (np.arange(len(sizes)) % 2).astype(np.int32)
    W = seeded_weights((len(sizes), ny, nx), rng)
    R = 20
    kmax = int(np.diff(ptr).max())
    for sh in ("box", "disk"):
        for thr in (0.5, 0.0):
            for vw in (None, seeded_views(vhp, rng, len(srcs), R)):
                for m in (1, 2, 3):
                    for w in (None, W):
                        for c in cs:
                            full = reference(c, occ, srcs, vw, ptr, kmax, m, thr, R, shape_of(vhp, sh), w, gmap)
                            quota = quotas_for(full, rng)
                            r = c.visibility_cover_quota_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), quota=quota,
                                                               m=m, weights=w, views=vw, kmax=kmax, group_map=gmap)
                            check_prefix(c, occ, srcs, vw, ptr, kmax, m, thr, R, shape_of(vhp, sh), w, gmap, quota,
                                         r, (n, sh, thr, vw is None, m, w is None))
    for c in cs:
        c.close()


def test_mixed_stopping_equals_each_problem_alone(ctx, vhp):
    rng = np.random.default_rng(5)
    nx, ny = 150, 110
    occ = np.stack([rect_map(nx, ny, 30, 50 + m, 3, 16) for m in range(2)])
    sizes = [30, 7, 0, 45, 12, 30, 1, 60, 25, 9, 40, 18]
    srcs, ptr = make_groups(rng, nx, ny, occ[0], sizes)
    gmap = (np.arange(len(sizes)) % 2).astype(np.int32)
    W = seeded_weights((len(sizes), ny, nx), rng)
    views = seeded_views(vhp, rng, len(srcs), 25)
    for vw, m in ((None, 1), (views, 2)):
        full = reference(ctx, occ, srcs, vw, ptr, 60, m, 0.5, 25, vhp.RANGE_DISK, W, gmap)
        quota = quotas_for(full, rng)
        r = ctx.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 25, vhp.RANGE_DISK, quota=quota, m=m, weights=W,
                                             views=vw, group_map=gmap)
        assert r["pick"].shape == (len(sizes), 60)  # kmax None: the largest group
        reasons = set()
        for q in range(len(sizes)):
            a, b = ptr[q], ptr[q + 1]
            one = ctx.visibility_cover_quota_batch(occ, srcs[a:b], [0, b - a], 0.5, 25, vhp.RANGE_DISK,
                                                   quota=quota[q:q + 1], m=m, weights=W[q:q + 1],
                                                   views=None if vw is None else vw[a:b], kmax=60,
                                                   group_map=gmap[q:q + 1])
            for key in ("pick", "gain", "npicked", "count", "total", "reached"):
                assert np.array_equal(r[key][q], one[key][0]), (q, key)
            reasons.add((bool(r["reached"][q]), int(r["npicked"][q]) == int(full["npicked"][q])))
        assert len(reasons) >= 2  # problems stopped both by the quota and by a gain of 0


def test_a_loop_of_thousands_of_rounds(ctx, vhp):
    """one problem of 4000 candidates of range 2 on a 400^2 map: full cover needs thousands of picks, so the graph
    loop runs thousands of rounds; each must be the m-fold call's, none skipped or repeated"""
    rng = np.random.default_rng(77)
    nx = ny = 400
    occ = rect_map(nx, ny, 200, 9, 3, 12)[None]
    srcs = np.stack([rng.integers(0, nx, 4000), rng.integers(0, ny, 4000)], 1).astype(np.int32)
    ptr = np.array([0, len(srcs)], np.int64)
    for m, w in ((1, None), (2, seeded_weights((1, ny, nx), rng))):
        u = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, len(srcs), m, 0.5, 2, vhp.RANGE_BOX, weights=w)
        r = ctx.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 2, vhp.RANGE_BOX, m=m, weights=w)
        assert r["npicked"][0] > 1000 and r["npicked"][0] == u["npicked"][0]
        for key in ("pick", "gain", "npicked", "count"):
            assert np.array_equal(r[key], u[key]), (m, key)
        assert int(r["total"][0]) == int(u["gain"].sum(dtype=np.uint64)) and not r["reached"][0]


def test_kmax(ctx, vhp):
    rng = np.random.default_rng(13)
    nx, ny = 90, 70
    occ = np.stack([rect_map(nx, ny, 10, 3, 3, 12)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [20, 0, 35])
    r = ctx.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 15, vhp.RANGE_DISK, kmax=0)
    assert r["pick"].shape == (3, 0) and not r["npicked"].any() and not r["count"].any() and not r["total"].any()
    assert not r["reached"].any()
    assert ctx.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 15, vhp.RANGE_DISK, quota=0, kmax=0)["reached"].all()
    for kmax in (1, 3, 7):
        u = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, kmax, 2, 0.5, 15, vhp.RANGE_DISK)
        r = ctx.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 15, vhp.RANGE_DISK, m=2, kmax=kmax)
        assert r["npicked"][1] == 0 and (r["npicked"][[0, 2]] == kmax).all()  # below what full cover needs
        for key in ("pick", "gain", "npicked", "count"):
            assert np.array_equal(r[key], u[key]), (kmax, key)
        assert not r["reached"].any()


@pytest.mark.parametrize("mode,thr,views", [(1, 0.5, False), (1, 0.0, False), (1, 0.5, True), (2, 0.5, False)])
def test_launches_do_not_depend_on_the_quota_kmax_or_rounds(vhp, ctx, mode, thr, views):
    import torch
    nsrc, R = 40, 16
    occ_t = dev_maps(torch, 1, 600, 600, 7)
    xy = torch.from_numpy(sources(nsrc, 600, 600, 8)).cuda()
    vw = torch.from_numpy(vhp.sensor_views(np.arange(nsrc) * 70.0, 90, R)).cuda() if views else None
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    pk = torch.empty((1, nsrc), dtype=torch.int32, device="cuda:0")
    cnt = torch.empty((1, 600, 600), dtype=torch.uint8, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        counts = set()
        for quota, kmax in ((0, 5), (1, 5), (U64_MAX, 1), (U64_MAX, nsrc), (300, 30)):
            q = torch.from_numpy(np.array([quota], np.uint64).view(np.int64)).cuda()
            fn = lambda: ctx.visibility_cover_quota_batch_dev(occ_t, xy, gptr, q, kmax, thr, R,  # noqa: E731
                                                              vhp.RANGE_DISK, m=2, pick_t=pk, count_t=cnt, views_t=vw)
            counts.add(launches_of(ctx, fn))
        assert len(counts) == 1, counts
        # the m-fold (or view) call of one round, whose rounds are 2 launches, plus the quota init and the graph
        ref = (lambda: ctx.visibility_cover_greedy_view_batch_dev(occ_t, xy, vw, gptr, 1, 2, thr, R, vhp.RANGE_DISK,
                                                                  pick_t=pk, count_t=cnt)) if views else \
            (lambda: ctx.visibility_cover_greedy_mfold_batch_dev(occ_t, xy, gptr, 1, 2, thr, R, vhp.RANGE_DISK,
                                                                 pick_t=pk, count_t=cnt))
        assert counts == {launches_of(ctx, ref) + 1}
    finally:
        ctx.set_grid_sweep(1)


def test_graph_is_fresh_after_the_buffers_grow(vhp):
    """a call, a larger call that grows the cover buffers, the first again, interleaved with the other cover calls:
    every result is unchanged (no graph holds a workspace pointer across calls)"""
    c = vhp.Context(0)
    rng = np.random.default_rng(31)
    small = (np.stack([rect_map(80, 60, 8, 1, 3, 10)]), 80, 60, [6, 9, 4])
    big = (np.stack([rect_map(300, 250, 60, 2, 3, 20)]), 300, 250, [200, 150, 120, 90])
    runs = []
    for occ, nx, ny, sizes in (small, big):
        srcs, ptr = make_groups(rng, nx, ny, occ[0], sizes)
        W = seeded_weights((len(sizes), ny, nx), rng)
        runs.append((occ, srcs, ptr, W, seeded_views(vhp, rng, len(srcs), 18)))

    def quota_call(i):
        occ, srcs, ptr, W, vw = runs[i]
        return c.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 18, vhp.RANGE_DISK, fraction=0.6, m=2, weights=W,
                                              views=vw)

    def others(i):
        occ, srcs, ptr, W, vw = runs[i]
        return (c.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, 5, 2, 0.5, 18, vhp.RANGE_DISK, weights=W),
                c.visibility_cover_greedy_view_batch(occ, srcs, vw, ptr, 5, 2, 0.0, 18, vhp.RANGE_BOX, weights=W),
                c.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, 4, 0.5, 18, vhp.RANGE_DISK, weights=W))

    a0, o0 = quota_call(0), others(0)
    b0 = quota_call(1)
    o1 = others(1)
    a1 = quota_call(0)
    b1 = quota_call(1)
    o2 = others(0)
    a2 = quota_call(0)
    for x, y in ((a0, a1), (a0, a2), (b0, b1)):
        for key in x:
            assert np.array_equal(x[key], y[key]), key
    for x, y in zip(o0, o2):
        for key in x:
            assert np.array_equal(x[key], y[key]), key
    assert o1[0]["npicked"].all() and a0["npicked"].any() and b0["npicked"].any()
    c.close()


def test_dev_equals_host(vhp):
    import torch
    rng = np.random.default_rng(8)
    nx, ny = 130, 96
    occ = np.stack([rect_map(nx, ny, 15, 60 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    srcs, ptr = make_groups(rng, nx, ny, occ[2], [4, 9, 0, 1, 40, 3, 25])
    gmap = np.array([2, 0, 1, 2, 1, 0, 1], np.int32)
    ng = len(ptr) - 1
    W = seeded_weights((ng, ny, nx), rng)
    stream = torch.cuda.Stream()
    c = vhp.torch_context(0, stream)
    occ_t, xy_t, ptr_t, gm_t, w_t = (torch.from_numpy(a).cuda() for a in (occ, srcs, ptr, gmap, W))
    torch.cuda.synchronize()
    for R, sh, thr, kmax, m, views in ((5, "disk", 0.5, 7, 2, True), (33, "box", 0.0, 40, 3, False),
                                       (60, "disk", 1e-9, 50, 1, True)):
        vw = seeded_views(vhp, rng, len(srcs), R) if views else None
        v_t = torch.from_numpy(vw).cuda() if views else None
        for w in (None, W):
            full = reference(c, occ, srcs, vw, ptr, kmax, m, thr, R, shape_of(vhp, sh), w, gmap)
            quota = quotas_for(full, rng)
            host = c.visibility_cover_quota_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), quota=quota, m=m,
                                                  weights=w, views=vw, kmax=kmax, group_map=gmap)
            with torch.cuda.stream(stream):
                q_t = torch.from_numpy(quota.view(np.int64)).cuda()
                pk = torch.full((ng, kmax), 5, dtype=torch.int32, device="cuda:0")
                gn = torch.full((ng, kmax), 5, dtype=torch.int64, device="cuda:0")
                npk = torch.full((ng,), 5, dtype=torch.int32, device="cuda:0")
                cnt = torch.full((ng, ny, nx), 5, dtype=torch.uint8, device="cuda:0")
                tot = torch.full((ng,), 5, dtype=torch.int64, device="cuda:0")
                c.visibility_cover_quota_batch_dev(occ_t, xy_t, ptr_t, q_t, kmax, thr, R, shape_of(vhp, sh), m=m,
                                                   pick_t=pk, gain_t=gn, npicked_t=npk, count_t=cnt, total_t=tot,
                                                   group_map_t=gm_t, weights_t=None if w is None else w_t,
                                                   views_t=v_t)
            c.synchronize()
            assert np.array_equal(pk.cpu().numpy(), host["pick"]), (R, sh, thr)
            assert np.array_equal(gn.cpu().numpy().view(np.uint64), host["gain"]), (R, sh, thr)
            assert np.array_equal(npk.cpu().numpy(), host["npicked"]), (R, sh, thr)
            assert np.array_equal(cnt.cpu().numpy(), host["count"]), (R, sh, thr)
            assert np.array_equal(tot.cpu().numpy().view(np.uint64), host["total"]), (R, sh, thr)
    c.close()


def test_two_4gb_runs_equal_one_problem_at_a_time(ctx, vhp):
    """8 weighted problems on 12000^2 maps with count: about 0.6 GB of device memory each, so the host form runs them
    in two runs, each with its own graph"""
    nx = ny = 12000
    rng = np.random.default_rng(43)
    occ = np.stack([rect_map(nx, ny, 3000, 200 + m, 10, 80) for m in range(2)]).astype(np.uint8)
    sizes = [5, 1, 9, 3, 6, 2, 7, 4]
    xy = np.stack([rng.integers(0, nx, sum(sizes)), rng.integers(0, ny, sum(sizes))], 1).astype(np.int32)
    xy[:3] = [(0, 0), (nx - 1, ny - 1), (6000, 0)]
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    gmap = (np.arange(8) % 2).astype(np.int32)
    W = rng.integers(0, 256, (8, ny, nx), dtype=np.uint8)
    R = 48
    views = seeded_views(vhp, rng, len(xy), R)
    quota = np.array([0, 1, 5000, 10**6, U64_MAX, 20000, 300000, 2], np.uint64)
    r = ctx.visibility_cover_quota_batch(occ, xy, ptr, 0.5, R, vhp.RANGE_DISK, quota=quota, m=2, weights=W,
                                         views=views, kmax=6, group_map=gmap)
    for q in range(8):
        a, b = ptr[q], ptr[q + 1]
        one = ctx.visibility_cover_quota_batch(occ, xy[a:b], [0, b - a], 0.5, R, vhp.RANGE_DISK, quota=quota[q:q + 1],
                                               m=2, weights=W[q:q + 1], views=views[a:b], kmax=6,
                                               group_map=gmap[q:q + 1])
        for key in ("pick", "gain", "npicked", "count", "total", "reached"):
            assert np.array_equal(r[key][q], one[key][0]), (q, key)
    assert r["npicked"][0] == 0 and (r["npicked"][2:] > 0).all()


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    good = np.array([(4, 1, 0, 0, 1), (4, 1, 1, 1, 1), (0, -1, 0, 1, 0)], np.int32)
    bad_views = [(-1, 1, 0, 0, 1), (5, 1, 0, 0, 1), (4, 0, 0, 0, 1), (4, 1, 0, 0, 0), (4, 32768, 0, 0, 1),
                 (4, 1, 0, 0, -32768)]
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2), dict(kmax=-1), dict(m=0), dict(m=256),
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),  # candidate outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                 # map out of range
        dict(group_ptr=[1, 3]),                                      # does not start at 0
        dict(group_ptr=[0, 2, 1, 3]),                                # decreasing
        dict(threshold=float("nan")),
    ] + [dict(views=np.array([good[0], v, good[2]], np.int32)) for v in bad_views]
    for b in bad:
        kw = dict(src_xy=srcs, group_ptr=[0, 3], threshold=0.5, radius=4, shape=vhp.RANGE_DISK, views=good, kmax=2,
                  m=2)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_quota_batch(occ, kw.pop("src_xy"), kw.pop("group_ptr"), kw.pop("threshold"),
                                           kw.pop("radius"), kw.pop("shape"), **kw)
        assert e.value.status == -1, b
        if "views" in b:
            assert b"view of candidate 1" in c.lib.vhp_last_error(c.h), b
        if "kmax" in b:
            assert b"vhp_visibility_cover_quota_batch: kmax < 0" in c.lib.vhp_last_error(c.h)
        r = c.visibility_cover_quota_batch(occ, srcs, [0, 3], 0.5, 4, vhp.RANGE_DISK, views=good, kmax=2, m=2)
        assert r["npicked"][0] == 2  # still works
    occ_u8 = np.ones((1, 20, 30), np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    npk = np.zeros(1, np.int32)
    one = vhp.CoverQuotaOut(None, None, npk.ctypes.data, None, None)
    tot = np.zeros(1, np.uint64)
    only_total = vhp.CoverQuotaOut(None, None, None, None, tot.ctypes.data)
    gp = np.array([0, 3], np.int64)
    q = np.array([5], np.uint64)
    fn = c.lib.vhp_visibility_cover_quota_batch
    args = lambda xy, views, ptr, quota, out: (c.h, vp(occ_u8), 1, 30, 20, vp(xy), views, vp(ptr), None, 1, 2, 4,  # noqa: E731,E501
                                                vhp.RANGE_BOX, 0.5, None, 2, quota, C.byref(out))
    assert fn(*args(srcs, None, gp, None, one)) == -1 and b"quota is NULL" in c.lib.vhp_last_error(c.h)
    none = vhp.CoverQuotaOut(None, None, None, None, None)
    assert fn(*args(srcs, None, gp, vp(q), none)) == -1 and b"no output" in c.lib.vhp_last_error(c.h)
    assert fn(*args(srcs, None, gp, vp(q), only_total)) == 0 and tot[0] >= 5  # total alone is an output
    big = np.array([0, 2**28], np.int64)
    assert fn(*args(srcs, vp(good), big, vp(q), one)) == -1 and b"2^28" in c.lib.vhp_last_error(c.h)
    # views NULL is the m-fold call; no problem needs no quota
    assert fn(*args(srcs, None, gp, vp(q), one)) == 0
    empty = np.array([0], np.int64)
    assert fn(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), None, vp(empty), None, 0, 2, 4, vhp.RANGE_BOX, 0.5, None, 2, None,
              C.byref(one)) == 0
    # the views are checked before any candidate is read: a bad view wins over a candidate outside the grid
    st = fn(*args(np.array([(1, 1), (30, 5), (7, 2)], np.int32),
                  vp(np.array([good[0], good[1], (9, 1, 0, 0, 1)], np.int32)), gp, vp(q), one))
    assert st == -1 and b"view of candidate 2" in c.lib.vhp_last_error(c.h)
    # the _dev form: bad arguments at once, a bad view through the device error flag (bit 3)
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    pk = torch.empty((2, 3), dtype=torch.int32, device=d)
    xy_ok = torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d)
    v_ok = torch.from_numpy(good).cuda()
    ptr_ok = torch.tensor([0, 1, 3], dtype=torch.int64, device=d)
    q_t = torch.tensor([3, 1000], dtype=torch.int64, device=d)
    for radius, shape, kmax, m, thr, quota in ((-1, vhp.RANGE_BOX, 3, 2, 0.5, q_t), (4, 2, 3, 2, 0.5, q_t),
                                               (4, vhp.RANGE_BOX, -1, 2, 0.5, q_t),
                                               (4, vhp.RANGE_BOX, 3, 2, float("nan"), q_t),
                                               (4, vhp.RANGE_BOX, 3, 0, 0.5, q_t), (4, vhp.RANGE_BOX, 3, 2, 0.5, None)):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_quota_batch_dev(occ_t, xy_ok, ptr_ok, quota, kmax, thr, radius, shape, m=m, pick_t=pk,
                                               views_t=v_ok)
        assert e.value.status == -1
    c.synchronize()
    with pytest.raises(vhp.VhpError) as e:
        c.visibility_cover_quota_batch_dev(occ_t, xy_ok, ptr_ok, q_t, 3, 0.5, 4, vhp.RANGE_BOX, m=2)
    assert b"no output" in c.lib.vhp_last_error(c.h)
    for thr in (0.5, 0.0):
        for v in bad_views:
            views = torch.tensor([good[0].tolist(), list(v), good[2].tolist()], dtype=torch.int32, device=d)
            c.visibility_cover_quota_batch_dev(occ_t, xy_ok, ptr_ok, q_t, 3, thr, 4, vhp.RANGE_BOX, m=2, pick_t=pk,
                                               views_t=views)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1 and b"view" in c.lib.vhp_last_error(c.h), (thr, v)
            c.visibility_cover_quota_batch_dev(occ_t, xy_ok, ptr_ok, q_t, 3, thr, 4, vhp.RANGE_BOX, m=2, pick_t=pk,
                                               views_t=v_ok)
            c.synchronize()
    # problem 0: (1, 1) with a quarter view of r = 4, 25 cells >= 3 after one pick; problem 1: (3, 1) sees its 7 x 5
    # written cells, then (2, 2) its own cell, and the quota of 1000 is not reached
    gn = torch.empty((2, 3), dtype=torch.int64, device=d)
    tt = torch.empty((2,), dtype=torch.int64, device=d)
    c.visibility_cover_quota_batch_dev(occ_t, xy_ok, ptr_ok, q_t, 3, 0.5, 4, vhp.RANGE_BOX, m=2, pick_t=pk,
                                       gain_t=gn, total_t=tt, views_t=v_ok)
    c.synchronize()
    assert pk.tolist() == [[0, -1, -1], [0, 1, -1]] and gn.tolist() == [[25, 0, 0], [35, 1, 0]]
    assert tt.tolist() == [25, 36]
    c.close()
