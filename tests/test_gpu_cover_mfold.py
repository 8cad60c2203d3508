"""Redundant (m-fold) greedy sensor placement (vhp_visibility_cover_greedy_mfold_batch) on the GPU: against the numpy
m-fold greedy of test_cover_mfold_cpu on the oracle's fields, against vhp_visibility_cover_greedy_weighted_batch at
m = 1, across the direct route and the fallback, against vhp_visibility_merge_range_batch on the picks, with gains
above 2^32, the _dev form against the host form, by launch count and on every error case.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

from conftest import rect_map
from test_cover_mfold_cpu import mgreedy
from test_cover_weighted_cpu import seeded_weights
from test_gpu_cover_weighted import problem_sets, shape_of
from test_gpu_merge import make_groups
from test_gpu_routes import dev_maps, launches_of, sources

pytestmark = pytest.mark.gpu
SHAPES = ("box", "disk")
THRS = (0.5, 1e-9, 0.0, -1.0)
MS = (1, 2, 3, 255)


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def mgreedy_all(psets, ks, m, shape, weights=None):
    """{k: [(pick, gain, npicked, count) per problem]}: one greedy of max(ks) rounds per problem, cut to each k (the
    first k rounds of a greedy are the greedy of k rounds)"""
    kmax = max(ks)
    res = {k: [] for k in ks}
    for q, sets in enumerate(psets):
        if sets:
            pick, gain, n, _ = mgreedy(sets, kmax, m, None if weights is None else weights[q])
        else:
            pick, gain, n = np.full(kmax, -1, np.int32), np.zeros(kmax, np.uint64), 0
        for k in ks:
            nk = min(n, k)
            cnt = np.zeros(shape, np.int64)
            for p in pick[:nk]:
                cnt += sets[p]
            res[k].append((pick[:k], gain[:k], nk, np.minimum(cnt, m).astype(np.uint8)))
    return res


def check(r, want, what):
    assert r["gain"].dtype == np.uint64 and r["count"].dtype == np.uint8
    for q, (pick, gain, n, cnt) in enumerate(want):
        assert np.array_equal(r["pick"][q], pick), (what, q, r["pick"][q], pick)
        assert np.array_equal(r["gain"][q], gain), (what, q, r["gain"][q], gain)
        assert r["npicked"][q] == n, (what, q)
        assert np.array_equal(r["count"][q], cnt), (what, q)


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny + 3)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    sizes = [0, 1, 2, 7, 33, 0, 2]  # empty groups, one candidate, duplicates (make_groups), on two maps
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 2 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)])
    weights = seeded_weights((len(sizes), ny, nx), rng)
    ks = (0, 1, 5, 40)  # 40: more than any group holds
    for R in (0, 1, 32, max(nx, ny) + 3):
        for sh in SHAPES:
            for thr in THRS:  # thr <= 0: the fallback
                psets = problem_sets(fields, srcs, ptr, thr, R, sh == "disk")
                for m in MS:
                    for w in (weights, None):
                        want = mgreedy_all(psets, ks, m, (ny, nx), w)
                        for k in ks:
                            r = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, k, m, thr, R,
                                                                        shape_of(vhp, sh), weights=w, group_map=gmap)
                            check(r, want[k], (shape, R, sh, thr, m, k, w is None))


def test_m_1_is_the_weighted_call(ctx, vhp):
    rng = np.random.default_rng(37)
    nx, ny = 150, 110
    occ = np.stack([rect_map(nx, ny, 30, 40 + m, 3, 16) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [50, 0, 1, 120, 9])
    gmap = np.array([0, 1, 0, 1, 1], np.int32)
    W = seeded_weights((len(ptr) - 1, ny, nx), rng)
    for R, sh, thr, k in ((20, "disk", 0.5, 9), (70, "box", 1e-9, 6), (12, "box", 0.0, 12), (200, "disk", -1.0, 3)):
        for w in (W, None):
            u = ctx.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh), weights=w,
                                                           group_map=gmap)
            r = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, k, 1, thr, R, shape_of(vhp, sh), weights=w,
                                                        group_map=gmap)
            what = (R, sh, thr, w is None)
            for key in ("pick", "gain", "npicked"):
                assert np.array_equal(r[key], u[key]), (what, key)
            assert r["count"].max() <= 1
            assert np.array_equal(r["count"] > 0, vhp.unpack_bits(u["covered"], nx)), what


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the box's size)
def test_routes_agree_and_match_library_fields(vhp, monkeypatch, n):
    rng = np.random.default_rng(n + 5)
    direct = vhp.Context(0)
    grid = vhp.Context(0)
    grid.set_grid_sweep(2)
    monkeypatch.setenv("VHP_SWEEP_IMPL", "naive")
    naive = vhp.Context(0)
    monkeypatch.delenv("VHP_SWEEP_IMPL")
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 10, 90 + m, 3, 14) for m in range(3)])
    nprob = 3 if n <= 12 else n // 50
    ptr = np.sort(np.concatenate([[0, n], rng.integers(0, n + 1, nprob - 1)])).astype(np.int64)
    srcs = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
    srcs[:4] = [(0, 0), (nx - 1, ny - 1), (31, 5), (32, 0)]
    gmap = rng.integers(0, 3, nprob).astype(np.int32)
    weights = seeded_weights((nprob, ny, nx), rng)
    fields = direct.visibility_batch(occ, srcs, src_map=np.repeat(gmap, np.diff(ptr)), dtype=vhp.F64)
    for R, sh, thr, k, m in ((16, "disk", 0.5, 6, 2), (40, "box", 1e-9, 4, 3), (7, "box", 0.0, 3, 2)):
        rs = [c.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, k, m, thr, R, shape_of(vhp, sh), weights=weights,
                                                    group_map=gmap) for c in (direct, grid, naive)]
        for r in rs[1:]:
            for key in ("pick", "gain", "npicked", "count"):
                assert np.array_equal(r[key], rs[0][key]), (n, R, sh, thr, key)
        if n <= 400:
            want = mgreedy_all(problem_sets(fields, srcs, ptr, thr, R, sh == "disk"), (k,), m, (ny, nx), weights)
            check(rs[0], want[k], (n, R, sh, thr, m))
    for c in (direct, grid, naive):
        c.close()


def test_count_is_the_range_merge_of_the_picks(ctx, vhp):
    rng = np.random.default_rng(11)
    nx, ny = 200, 150
    occ = np.stack([rect_map(nx, ny, 40, 30 + m, 3, 20) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [60, 1, 0, 90])
    gmap = np.array([0, 1, 0, 1], np.int32)
    W = seeded_weights((4, ny, nx), rng)
    for R, sh, thr, m in ((25, "disk", 0.5, 2), (60, "box", 0.0, 3), (40, "disk", 0.5, 255)):
        r = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, 12, m, thr, R, shape_of(vhp, sh), weights=W,
                                                    group_map=gmap)
        picks = [srcs[ptr[q] + r["pick"][q][:r["npicked"][q]]] for q in range(4)]
        assert all(len(set(r["pick"][q][:r["npicked"][q]].tolist())) == r["npicked"][q] for q in range(4))
        pptr = np.concatenate([[0], np.cumsum([len(p) for p in picks])]).astype(np.int64)
        mg = ctx.visibility_merge_range_batch(occ, np.concatenate(picks), pptr, thr, R, shape_of(vhp, sh),
                                              group_map=gmap, outputs=("count",))
        cnt = np.minimum(mg["count"], m)
        assert np.array_equal(r["count"], cnt.astype(np.uint8)), (R, sh, thr, m)
        assert (np.diff(r["gain"].astype(np.int64), axis=1) <= 0).all()
        assert np.array_equal(r["gain"].sum(1), (W.astype(np.uint64) * cnt.astype(np.uint64)).sum((1, 2)))


def test_gains_above_2_pow_32(ctx, vhp):
    """an empty 4200^2 map, every weight 255, whole-map boxes: (0, 0) sees the whole map, (0, 3000) all but row 0
    (every written cell of an empty map is lit).  Its duplicate is picked after it when m = 3, not when m = 2"""
    nx = ny = 4200
    occ = np.ones((1, ny, nx), np.uint8)
    xy = np.array([(0, 3000), (0, 3000), (0, 0)], np.int32)
    ptr = np.array([0, 3], np.int64)
    W = np.full((1, ny, nx), 255, np.uint8)
    N = nx * ny
    for thr in (0.5, 0.0):
        for m, pick, gain, top in ((2, [2, 0, -1], [255 * N, 255 * (N - nx), 0], 2),
                                   (3, [2, 0, 1], [255 * N, 255 * (N - nx), 255 * (N - nx)], 3)):
            r = ctx.visibility_cover_greedy_mfold_batch(occ, xy, ptr, 3, m, thr, nx, vhp.RANGE_BOX, weights=W)
            assert r["pick"][0].tolist() == pick and r["gain"][0].tolist() == gain, (thr, m)
            assert r["gain"][0, 1] > 2**32 and r["npicked"][0] == 3 - pick.count(-1)
            assert (r["count"][0, 0] == 1).all() and (r["count"][0, 1:] == top).all(), (thr, m)


def test_dev_equals_host(vhp):
    import torch
    rng = np.random.default_rng(6)
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
    for R, sh, thr, k, m in ((5, "disk", 0.5, 7, 2), (33, "box", 0.0, 3, 3), (60, "disk", 1e-9, 50, 255)):
        for w in (None, W):
            host = c.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, k, m, thr, R, shape_of(vhp, sh), weights=w,
                                                         group_map=gmap)
            with torch.cuda.stream(stream):
                pk = torch.full((ng, k), 5, dtype=torch.int32, device="cuda:0")
                gn = torch.full((ng, k), 5, dtype=torch.int64, device="cuda:0")
                npk = torch.full((ng,), 5, dtype=torch.int32, device="cuda:0")
                cnt = torch.full((ng, ny, nx), 5, dtype=torch.uint8, device="cuda:0")
                c.visibility_cover_greedy_mfold_batch_dev(occ_t, xy_t, ptr_t, k, m, thr, R, shape_of(vhp, sh),
                                                          pick_t=pk, gain_t=gn, npicked_t=npk, count_t=cnt,
                                                          group_map_t=gm_t, weights_t=None if w is None else w_t)
            c.synchronize()
            assert np.array_equal(pk.cpu().numpy(), host["pick"]), (R, sh, thr)
            assert np.array_equal(gn.cpu().numpy().view(np.uint64), host["gain"]), (R, sh, thr)
            assert np.array_equal(npk.cpu().numpy(), host["npicked"]), (R, sh, thr)
            assert np.array_equal(cnt.cpu().numpy(), host["count"]), (R, sh, thr)
    c.close()


@pytest.mark.parametrize("mode,thr,k,count,want", [
    (1, 0.5, 3, True, 10),    # table + box sweep + weight plane + init + 3 applies + 2 updates + count
    (1, 0.5, 3, False, 9),    # no count output: no count kernel
    (1, 0.5, 10, True, 14),   # rounds = min(k, nsrc) = 5
    (1, 0.5, 0, True, 1),     # k = 0: the table only (count zeroed by a memset)
    (1, 0.0, 3, True, 11),    # fallback: windowed kernel + fold
    (1, 0.0, 3, False, 10),
    (2, 0.5, 3, True, 22),    # grid mode forced: sanitised pairs + 2 grid kernels per pair + crop, then the fold
])
def test_routes_by_launch_count(vhp, ctx, mode, thr, k, count, want):
    import torch
    nsrc, R = 5, 16
    occ_t = dev_maps(torch, 1, 1000, 1000, 7)
    xy = torch.from_numpy(sources(nsrc, 1000, 1000, 8)).cuda()
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    pk = torch.empty((1, max(k, 1)), dtype=torch.int32, device="cuda:0")
    cnt = torch.empty((1, 1000, 1000), dtype=torch.uint8, device="cuda:0") if count else None
    w = torch.ones((1, 1000, 1000), dtype=torch.uint8, device="cuda:0")
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        call = lambda: ctx.visibility_cover_greedy_mfold_batch_dev(occ_t, xy, gptr, k, 2, thr, R,  # noqa: E731
                                                                   vhp.RANGE_DISK, pick_t=pk, count_t=cnt,
                                                                   weights_t=w)
        assert launches_of(ctx, call) == want
        if count and k == 0:
            ctx.synchronize()
            assert not cnt.any()
    finally:
        ctx.set_grid_sweep(1)


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2), dict(shape=-1), dict(k=-1), dict(m=0), dict(m=256),
        dict(m=-1), dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),  # candidate outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                             # map out of range
        dict(group_ptr=[1, 3]),                                                  # does not start at 0
        dict(group_ptr=[0, 2, 1, 3]),                                            # decreasing
        dict(threshold=float("nan")),
    ]
    for b in bad:
        kw = dict(src_xy=srcs, group_ptr=[0, 3], k=2, m=2, threshold=0.5, radius=4, shape=vhp.RANGE_DISK)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_mfold_batch(occ, kw.pop("src_xy"), kw.pop("group_ptr"), kw.pop("k"),
                                                  kw.pop("m"), kw.pop("threshold"), kw.pop("radius"), kw.pop("shape"),
                                                  **kw)
        assert e.value.status == -1, b
        r = c.visibility_cover_greedy_mfold_batch(occ, srcs, [0, 3], 2, 2, 0.5, 4, vhp.RANGE_DISK)  # still works
        assert r["npicked"][0] == 2
    for m in (0, 256):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_mfold_batch(occ, srcs, [0, 3], 2, m, 0.5, 4, vhp.RANGE_DISK)
        assert b"m outside [1, 255]" in c.lib.vhp_last_error(c.h)
    occ_u8 = np.ones((1, 20, 30), np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    none = vhp.CoverMfoldOut(None, None, None, None)
    gp = np.array([0, 3], np.int64)
    st = c.lib.vhp_visibility_cover_greedy_mfold_batch(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), vp(gp), None, 1, 2, 4,
                                                       vhp.RANGE_BOX, 0.5, None, 2, C.byref(none))
    assert st == -1 and b"no output" in c.lib.vhp_last_error(c.h)
    # 2^28 candidates: rejected on group_ptr[nprob] before a candidate is read (srcs holds 3)
    npk = np.zeros(1, np.int32)
    one = vhp.CoverMfoldOut(None, None, npk.ctypes.data, None)
    big = np.array([0, 2**28], np.int64)
    st = c.lib.vhp_visibility_cover_greedy_mfold_batch(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), vp(big), None, 1, 2, 4,
                                                       vhp.RANGE_BOX, 0.5, None, 2, C.byref(one))
    assert st == -1 and b"2^28" in c.lib.vhp_last_error(c.h)
    r = c.visibility_cover_greedy_mfold_batch(occ, srcs, [0, 3], 0, 2, 0.5, 4, vhp.RANGE_DISK)  # k = 0 is valid
    assert r["pick"].shape == (1, 0) and r["gain"].dtype == np.uint64 and r["npicked"][0] == 0
    assert r["count"].shape == (1, 20, 30) and not r["count"].any()
    # the _dev form: bad arguments at once, a bad candidate / group layout through the device error flag
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    pk = torch.empty((2, 3), dtype=torch.int32, device=d)
    xy_ok = torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d)
    ptr_ok = torch.tensor([0, 1, 3], dtype=torch.int64, device=d)
    for radius, shape, k, m, thr in ((-1, vhp.RANGE_BOX, 3, 2, 0.5), (16384, vhp.RANGE_BOX, 3, 2, 0.5),
                                     (4, 2, 3, 2, 0.5), (4, vhp.RANGE_BOX, -1, 2, 0.5),
                                     (4, vhp.RANGE_BOX, 3, 2, float("nan")), (4, vhp.RANGE_BOX, 3, 0, 0.5),
                                     (4, vhp.RANGE_BOX, 3, 256, 0.5)):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_mfold_batch_dev(occ_t, xy_ok, ptr_ok, k, m, thr, radius, shape, pick_t=pk)
        assert e.value.status == -1
    with pytest.raises(vhp.VhpError) as e:
        c.visibility_cover_greedy_mfold_batch_dev(occ_t, xy_ok, ptr_ok, 3, 2, 0.5, 4, vhp.RANGE_BOX)
    assert e.value.status == -1
    # nsrc = 2^28 in the _dev form: rejected before any launch
    c.synchronize()
    before = c.launches
    dout = vhp.CoverMfoldOut(pk.data_ptr(), None, None, None)
    st = c.lib.vhp_visibility_cover_greedy_mfold_batch_dev(c.h, occ_t.data_ptr(), 1, 30, 20, xy_ok.data_ptr(),
                                                           ptr_ok.data_ptr(), None, 2, 2**28, 3, 4, vhp.RANGE_BOX,
                                                           0.5, None, 2, C.byref(dout))
    assert st == -1 and b"2^28" in c.lib.vhp_last_error(c.h) and c.launches == before
    c.synchronize()
    for thr in (0.5, 0.0):
        for xy, ptr in (([(1, 1), (31, 1), (2, 2)], [0, 1, 3]), ([(1, 1), (3, 1), (2, 2)], [0, 2, 1])):
            c.visibility_cover_greedy_mfold_batch_dev(occ_t, torch.tensor(xy, dtype=torch.int32, device=d),
                                                      torch.tensor(ptr, dtype=torch.int64, device=d), 3, 2, thr, 4,
                                                      vhp.RANGE_BOX, pick_t=pk)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1, (thr, xy, ptr)
    gn = torch.empty((2, 3), dtype=torch.int64, device=d)
    c.visibility_cover_greedy_mfold_batch_dev(occ_t, xy_ok, ptr_ok, 3, 2, 0.5, 4, vhp.RANGE_BOX, pick_t=pk,
                                              gain_t=gn)
    c.synchronize()
    # problem 0: (1, 1) covers its 5 x 5 written cells; problem 1: (2, 2) covers 36 cells, then (3, 1) all of its 35,
    # every one of them covered fewer than 2 times
    assert pk.tolist() == [[0, -1, -1], [1, 0, -1]]
    assert gn.tolist() == [[25, 0, 0], [36, 35, 0]]
    c.close()
