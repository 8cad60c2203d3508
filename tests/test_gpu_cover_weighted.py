"""Weighted greedy sensor placement (vhp_visibility_cover_greedy_weighted_batch) on the GPU: against the numpy weighted
greedy of test_cover_weighted_cpu on the oracle's fields, against vhp_visibility_cover_greedy_batch (no weights, and
weights in {0, 1} as its target), across the direct route and the fallback, against vhp_visibility_merge_range_batch
on the picks, with gains above 2^32, beyond the one-CTA kernel's whole-map limit, by launch count and on every error
case.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

from conftest import rect_map
from test_cover_cpu import cover_set
from test_cover_weighted_cpu import seeded_weights, wgreedy
from test_gpu_merge import make_groups
from test_gpu_routes import dev_maps, launches_of, sources

pytestmark = pytest.mark.gpu
SHAPES = ("box", "disk")
THRS = (0.5, 1e-9, 0.0, -1.0)


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


def problem_sets(fields, srcs, ptr, thr, R, disk):
    return [[cover_set(f, int(sx), int(sy), thr, R, disk) for f, (sx, sy) in zip(fields[a:b], srcs[a:b])]
            for a, b in zip(ptr[:-1], ptr[1:])]


def wgreedy_all(psets, k, shape, weights=None):
    """pick, gain, npicked, covered (bool) per problem"""
    return [wgreedy(sets, k, None if weights is None else weights[q]) if sets else
            (np.full(k, -1, np.int32), np.zeros(k, np.uint64), 0, np.zeros(shape, bool))
            for q, sets in enumerate(psets)]


def check(vhp, r, want, nx, what):
    assert r["gain"].dtype == np.uint64
    for q, (pick, gain, n, U) in enumerate(want):
        assert np.array_equal(r["pick"][q], pick), (what, q, r["pick"][q], pick)
        assert np.array_equal(r["gain"][q], gain), (what, q, r["gain"][q], gain)
        assert r["npicked"][q] == n, (what, q)
        assert np.array_equal(vhp.unpack_bits(r["covered"][q], nx), U), (what, q)
    assert not (r["covered"] & ~vhp.pack_bits(np.ones(r["covered"].shape[1:2] + (nx,), bool))).any()  # bits >= nx


def same(r, u, what):
    """the weighted call's outputs equal the cover call's, gains as integers"""
    assert np.array_equal(r["pick"], u["pick"]), what
    assert np.array_equal(r["gain"], u["gain"].astype(np.uint64)), what
    assert np.array_equal(r["npicked"], u["npicked"]), what
    assert np.array_equal(r["covered"], u["covered"]), what


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny + 2)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    sizes = [0, 1, 2, 7, 33, 0, 2]  # empty groups, one candidate, duplicates (make_groups), on two maps
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 2 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)])
    weights = seeded_weights((len(sizes), ny, nx), rng)
    for R in (0, 1, 31, 32, 33, max(nx, ny) + 3):
        for sh in SHAPES:
            for thr in THRS:  # thr <= 0: the fallback
                psets = problem_sets(fields, srcs, ptr, thr, R, sh == "disk")
                for k in (0, 1, 5, 40):  # 40: more than any group holds
                    for w in (weights, None):
                        want = wgreedy_all(psets, k, (ny, nx), w)
                        r = ctx.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh),
                                                                       weights=w, group_map=gmap)
                        check(vhp, r, want, nx, (shape, R, sh, thr, k, w is None))


def test_identities_with_the_cover_call(ctx, vhp):
    """no weights = the cover call without a target; weights in {0, 1} = the cover call with them as its target"""
    rng = np.random.default_rng(31)
    nx, ny = 150, 110
    occ = np.stack([rect_map(nx, ny, 30, 40 + m, 3, 16) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [50, 0, 1, 120, 9])
    gmap = np.array([0, 1, 0, 1, 1], np.int32)
    T = rng.random((len(ptr) - 1, ny, nx)) < 0.4
    for R, sh, thr, k in ((20, "disk", 0.5, 9), (70, "box", 1e-9, 6), (12, "box", 0.0, 12), (200, "disk", -1.0, 3)):
        u = ctx.visibility_cover_greedy_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh), group_map=gmap)
        r = ctx.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh), group_map=gmap)
        same(r, u, (R, sh, thr, "no weights"))
        u = ctx.visibility_cover_greedy_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh), group_map=gmap, target=T)
        r = ctx.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh),
                                                       weights=T.astype(np.uint8), group_map=gmap)
        same(r, u, (R, sh, thr, "binary weights"))


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the box's size)
def test_routes_agree_and_match_library_fields(vhp, monkeypatch, n):
    rng = np.random.default_rng(n + 1)
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
    for R, sh, thr, k in ((16, "disk", 0.5, 6), (40, "box", 1e-9, 4), (7, "box", 0.0, 3)):
        rs = [c.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh), weights=weights,
                                                       group_map=gmap) for c in (direct, grid, naive)]
        for r in rs[1:]:
            for key in ("pick", "gain", "npicked", "covered"):
                assert np.array_equal(r[key], rs[0][key]), (n, R, sh, thr, key)
        if n <= 400:
            want = wgreedy_all(problem_sets(fields, srcs, ptr, thr, R, sh == "disk"), k, (ny, nx), weights)
            check(vhp, rs[0], want, nx, (n, R, sh, thr))
    for c in (direct, grid, naive):
        c.close()


def test_covered_is_the_range_merge_of_the_picks(ctx, vhp):
    rng = np.random.default_rng(9)
    nx, ny = 200, 150
    occ = np.stack([rect_map(nx, ny, 40, 30 + m, 3, 20) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [60, 1, 0, 90])
    gmap = np.array([0, 1, 0, 1], np.int32)
    W = seeded_weights((4, ny, nx), rng)
    for R, sh, thr in ((25, "disk", 0.5), (60, "box", 0.0)):
        r = ctx.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, 12, thr, R, shape_of(vhp, sh), weights=W,
                                                       group_map=gmap)
        picks = [srcs[ptr[q] + r["pick"][q][:r["npicked"][q]]] for q in range(4)]
        pptr = np.concatenate([[0], np.cumsum([len(p) for p in picks])]).astype(np.int64)
        m = ctx.visibility_merge_range_batch(occ, np.concatenate(picks), pptr, thr, R, shape_of(vhp, sh),
                                             group_map=gmap, outputs=("count",))
        U = m["count"] > 0
        assert np.array_equal(vhp.unpack_bits(r["covered"], nx), U), (R, sh, thr)
        assert (np.diff(r["gain"].astype(np.int64), axis=1) <= 0).all()
        assert np.array_equal(r["gain"].sum(1), (W.astype(np.uint64) * U).sum((1, 2))), (R, sh, thr)


def test_gains_above_2_pow_32(ctx, vhp):
    """an empty 4200^2 map, every weight 255, whole-map boxes: gains up to 255 * 4200^2 > 2^32, against the closed
    form 255 * |writes & box| (every written cell of an empty map is lit)"""
    nx = ny = 4200
    occ = np.ones((1, ny, nx), np.uint8)
    # problem 0 picks (0, 3000) (all but row 0), then (9, 9) and (2100, 2100) add nothing; problem 1 picks (0, 0)
    # (the whole map); problem 2 picks (3000, 0) (all but column 0)
    xy = np.array([(9, 9), (2100, 2100), (0, 3000), (0, 0), (3000, 0)], np.int32)
    ptr = np.array([0, 3, 4, 5], np.int64)
    W = np.full((3, ny, nx), 255, np.uint8)
    N = nx * ny
    for thr in (0.5, 0.0):
        r = ctx.visibility_cover_greedy_weighted_batch(occ, xy, ptr, 3, thr, nx, vhp.RANGE_BOX, weights=W)
        assert r["pick"].tolist() == [[2, -1, -1], [0, -1, -1], [0, -1, -1]], thr
        assert r["gain"][:, 0].tolist() == [255 * (N - nx), 255 * N, 255 * (N - ny)], thr
        assert r["gain"][:, 0].min() > 2**32 and not r["gain"][:, 1:].any()
        assert r["npicked"].tolist() == [1, 1, 1]
        cov = vhp.unpack_bits(r["covered"], nx)
        assert cov[0, 1:].all() and not cov[0, 0].any() and cov[1].all()
        assert cov[2][:, 1:].all() and not cov[2][:, 0].any()


def test_beyond_one_cta_map_limit(vhp):
    """12000 x 12000, R = 40: against the weighted greedy over sets built from visibility_window_batch_dev's fp64
    windows"""
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
    W = rng.integers(0, 256, (1, ny, nx), dtype=np.uint8)
    W[0, 5990:6010, :] = 0
    w_t = torch.from_numpy(W).cuda()
    Wf = W[0].reshape(-1).astype(np.int64)
    R, k, P = 40, 10, 81
    win = torch.empty((len(xy), P, P), dtype=torch.float64, device="cuda:0")
    c.visibility_window_batch_dev(occ_t, xy_t, R, win)
    c.synchronize()
    win = win.cpu().numpy()
    v, u = np.mgrid[-R:R + 1, -R:R + 1]
    for sh in SHAPES:
        for thr in (0.5, 0.0):
            sets = []
            for w, (sx, sy) in zip(win, xy):
                x, y = sx + u, sy + v
                m = (x >= 0) & (x < nx) & (y >= 0) & (y < ny) & (w >= thr)
                m &= ~((x == 0) & (sx != 0)) & ~((y == 0) & (sy != 0))
                if sh == "disk":
                    m &= u * u + v * v <= R * R
                sets.append(set((y[m].astype(np.int64) * nx + x[m]).tolist()))
            U, pick, gain = set(), [], []
            for _ in range(k):
                g = [int(Wf[np.fromiter(s - U, np.int64)].sum()) for s in sets]
                p = int(np.argmax(g))
                if g[p] == 0:
                    break
                pick.append(p)
                gain.append(g[p])
                U |= sets[p]
            pk = torch.full((1, k), 9, dtype=torch.int32, device="cuda:0")
            gn = torch.full((1, k), 9, dtype=torch.int64, device="cuda:0")
            npk = torch.full((1,), 9, dtype=torch.int32, device="cuda:0")
            cov = torch.full((1, ny, (nx + 31) // 32), 9, dtype=torch.int32, device="cuda:0")
            torch.cuda.synchronize()
            c.visibility_cover_greedy_weighted_batch_dev(occ_t, xy_t, ptr_t, k, thr, R, shape_of(vhp, sh),
                                                         pick_t=pk, gain_t=gn, npicked_t=npk, covered_t=cov,
                                                         weights_t=w_t)
            c.synchronize()
            n = len(pick)
            assert pk[0].tolist() == pick + [-1] * (k - n), (sh, thr)
            assert gn[0].tolist() == gain + [0] * (k - n), (sh, thr)
            assert npk.item() == n
            cells = np.flatnonzero(vhp.unpack_bits(cov[0].cpu().numpy().view(np.uint32), nx))
            assert np.array_equal(cells, np.array(sorted(U), np.int64)), (sh, thr)
            del pk, gn, npk, cov
    c.close()


def test_dev_equals_host(vhp):
    import torch
    rng = np.random.default_rng(4)
    nx, ny = 130, 96
    occ = np.stack([rect_map(nx, ny, 15, 60 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    srcs, ptr = make_groups(rng, nx, ny, occ[2], [4, 9, 0, 1, 40, 3])
    gmap = np.array([2, 0, 1, 2, 1, 0], np.int32)
    ng, nw = len(ptr) - 1, (nx + 31) // 32
    W = seeded_weights((ng, ny, nx), rng)
    stream = torch.cuda.Stream()
    c = vhp.torch_context(0, stream)
    occ_t, xy_t, ptr_t, gm_t, w_t = (torch.from_numpy(a).cuda() for a in (occ, srcs, ptr, gmap, W))
    torch.cuda.synchronize()
    for R, sh, thr, k in ((5, "disk", 0.5, 7), (33, "box", 0.0, 3), (60, "disk", 1e-9, 50)):
        for w in (None, W):
            host = c.visibility_cover_greedy_weighted_batch(occ, srcs, ptr, k, thr, R, shape_of(vhp, sh), weights=w,
                                                            group_map=gmap)
            with torch.cuda.stream(stream):
                pk = torch.full((ng, k), 5, dtype=torch.int32, device="cuda:0")
                gn = torch.full((ng, k), 5, dtype=torch.int64, device="cuda:0")
                npk = torch.full((ng,), 5, dtype=torch.int32, device="cuda:0")
                cov = torch.full((ng, ny, nw), 5, dtype=torch.int32, device="cuda:0")
                c.visibility_cover_greedy_weighted_batch_dev(occ_t, xy_t, ptr_t, k, thr, R, shape_of(vhp, sh),
                                                             pick_t=pk, gain_t=gn, npicked_t=npk, covered_t=cov,
                                                             group_map_t=gm_t, weights_t=None if w is None else w_t)
            c.synchronize()
            assert np.array_equal(pk.cpu().numpy(), host["pick"]), (R, sh, thr)
            assert np.array_equal(gn.cpu().numpy().view(np.uint64), host["gain"]), (R, sh, thr)
            assert np.array_equal(npk.cpu().numpy(), host["npicked"]), (R, sh, thr)
            assert np.array_equal(cov.cpu().numpy().view(np.uint32), host["covered"]), (R, sh, thr)
    c.close()


@pytest.mark.parametrize("mode,thr,k,weights,want", [
    (1, 0.5, 3, True, 9),     # table + box sweep + weight plane + init + 3 applies + 2 updates
    (1, 0.5, 3, False, 9),    # no weights: the weight plane of ones all the same
    (1, 0.5, 10, True, 13),   # rounds = min(k, nsrc) = 5
    (1, 0.5, 0, True, 1),     # k = 0: the table only
    (1, 0.0, 3, True, 10),    # fallback: windowed kernel + fold
    (2, 0.5, 3, True, 21),    # grid mode forced: sanitised pairs + 2 grid kernels per pair + crop, then the fold
])
def test_routes_by_launch_count(vhp, ctx, mode, thr, k, weights, want):
    import torch
    nsrc, R = 5, 16
    occ_t = dev_maps(torch, 1, 1000, 1000, 7)
    xy = torch.from_numpy(sources(nsrc, 1000, 1000, 8)).cuda()
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    pk = torch.empty((1, max(k, 1)), dtype=torch.int32, device="cuda:0")
    w = torch.ones((1, 1000, 1000), dtype=torch.uint8, device="cuda:0") if weights else None
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        call = lambda: ctx.visibility_cover_greedy_weighted_batch_dev(occ_t, xy, gptr, k, thr, R,  # noqa: E731
                                                                      vhp.RANGE_DISK, pick_t=pk, weights_t=w)
        assert launches_of(ctx, call) == want
    finally:
        ctx.set_grid_sweep(1)


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2), dict(shape=-1), dict(k=-1),
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),  # candidate outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                    # map out of range
        dict(group_ptr=[1, 3]),                                         # does not start at 0
        dict(group_ptr=[0, 2, 1, 3]),                                   # decreasing
        dict(threshold=float("nan")),
    ]
    for b in bad:
        kw = dict(src_xy=srcs, group_ptr=[0, 3], k=2, threshold=0.5, radius=4, shape=vhp.RANGE_DISK)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_weighted_batch(occ, kw.pop("src_xy"), kw.pop("group_ptr"), kw.pop("k"),
                                                     kw.pop("threshold"), kw.pop("radius"), kw.pop("shape"), **kw)
        assert e.value.status == -1, b
        r = c.visibility_cover_greedy_weighted_batch(occ, srcs, [0, 3], 2, 0.5, 4, vhp.RANGE_DISK)  # still works
        assert r["npicked"][0] == 2
    occ_u8 = np.ones((1, 20, 30), np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    none = vhp.CoverWeightedOut(None, None, None, None)
    gp = np.array([0, 3], np.int64)
    st = c.lib.vhp_visibility_cover_greedy_weighted_batch(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), vp(gp), None, 1, 2, 4,
                                                          vhp.RANGE_BOX, 0.5, None, C.byref(none))
    assert st == -1 and b"no output" in c.lib.vhp_last_error(c.h)
    # 2^28 candidates: rejected on group_ptr[nprob] before a candidate is read (srcs holds 3)
    npk = np.zeros(1, np.int32)
    one = vhp.CoverWeightedOut(None, None, npk.ctypes.data, None)
    big = np.array([0, 2**28], np.int64)
    st = c.lib.vhp_visibility_cover_greedy_weighted_batch(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), vp(big), None, 1, 2,
                                                          4, vhp.RANGE_BOX, 0.5, None, C.byref(one))
    assert st == -1 and b"2^28" in c.lib.vhp_last_error(c.h)
    r = c.visibility_cover_greedy_weighted_batch(occ, srcs, [0, 3], 0, 0.5, 4, vhp.RANGE_DISK)  # k = 0 is valid
    assert r["pick"].shape == (1, 0) and r["gain"].dtype == np.uint64 and r["npicked"][0] == 0
    assert not r["covered"].any()
    # the _dev form: bad arguments at once, a bad candidate / group layout through the device error flag
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    pk = torch.empty((2, 3), dtype=torch.int32, device=d)
    xy_ok = torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d)
    ptr_ok = torch.tensor([0, 1, 3], dtype=torch.int64, device=d)
    for radius, shape, k, thr in ((-1, vhp.RANGE_BOX, 3, 0.5), (16384, vhp.RANGE_BOX, 3, 0.5), (4, 2, 3, 0.5),
                                  (4, vhp.RANGE_BOX, -1, 0.5), (4, vhp.RANGE_BOX, 3, float("nan"))):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_greedy_weighted_batch_dev(occ_t, xy_ok, ptr_ok, k, thr, radius, shape, pick_t=pk)
        assert e.value.status == -1
    with pytest.raises(vhp.VhpError) as e:
        c.visibility_cover_greedy_weighted_batch_dev(occ_t, xy_ok, ptr_ok, 3, 0.5, 4, vhp.RANGE_BOX)
    assert e.value.status == -1
    # nsrc = 2^28 in the _dev form: rejected before any launch
    c.synchronize()
    before = c.launches
    dout = vhp.CoverWeightedOut(pk.data_ptr(), None, None, None)
    st = c.lib.vhp_visibility_cover_greedy_weighted_batch_dev(c.h, occ_t.data_ptr(), 1, 30, 20, xy_ok.data_ptr(),
                                                              ptr_ok.data_ptr(), None, 2, 2**28, 3, 4, vhp.RANGE_BOX,
                                                              0.5, None, C.byref(dout))
    assert st == -1 and b"2^28" in c.lib.vhp_last_error(c.h) and c.launches == before
    c.synchronize()
    for thr in (0.5, 0.0):
        for xy, ptr in (([(1, 1), (31, 1), (2, 2)], [0, 1, 3]), ([(1, 1), (3, 1), (2, 2)], [0, 2, 1])):
            c.visibility_cover_greedy_weighted_batch_dev(occ_t, torch.tensor(xy, dtype=torch.int32, device=d),
                                                         torch.tensor(ptr, dtype=torch.int64, device=d), 3, thr, 4,
                                                         vhp.RANGE_BOX, pick_t=pk)
            with pytest.raises(vhp.VhpError) as e:
                c.synchronize()
            assert e.value.status == -1, (thr, xy, ptr)
    gn = torch.empty((2, 3), dtype=torch.int64, device=d)
    c.visibility_cover_greedy_weighted_batch_dev(occ_t, xy_ok, ptr_ok, 3, 0.5, 4, vhp.RANGE_BOX, pick_t=pk, gain_t=gn)
    c.synchronize()
    assert pk.tolist() == [[0, -1, -1], [1, 0, -1]]  # (2, 2) covers 36 cells, (3, 1) 35, 5 of them new after it
    assert gn.tolist() == [[25, 0, 0], [36, 5, 0]]  # (1, 1): 5 x 5 written cells
    c.close()
