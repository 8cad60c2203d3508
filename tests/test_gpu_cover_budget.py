"""Budgeted sensor placement (vhp_visibility_cover_budget_batch) on the GPU: the numpy budget greedy on the oracle's
fields on every route and warp size, the identities with the view / m-fold call and the quota call, Farey near-ties
of the ratio, problems stopping for different reasons in one call, a loop of thousands of rounds, launch counts, graph
freshness across calls that grow the buffers, the _dev form against the host form, a host call over two 4 GB runs, and
every error case.  Every comparison is exact."""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import rect_map
from test_cover_budget_cpu import bgreedy
from test_cover_view_cpu import view_sets
from test_cover_weighted_cpu import seeded_weights
from test_gpu_cover_quota import reference
from test_gpu_cover_view import contexts, seeded_views
from test_gpu_cover_weighted import problem_sets, shape_of
from test_gpu_merge import make_groups
from test_gpu_routes import dev_maps, launches_of, sources

pytestmark = pytest.mark.gpu
U64_MAX = np.iinfo(np.uint64).max
KEYS = ("pick", "gain", "npicked", "count", "total", "spent", "single", "single_gain")


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def check(r, psets, ptr, kmax, m, cost, budget, quota, W, shape, what):
    for q, sets in enumerate(psets):
        a = ptr[q]
        w = None if W is None else W[q]
        qq = None if quota is None else int(quota[q])
        if sets:
            want = bgreedy(sets, kmax, m, cost[a:a + len(sets)], int(budget[q]), qq, w)
        else:
            want = (np.full(kmax, -1, np.int32), np.zeros(kmax, np.uint64), 0, np.zeros(shape, np.uint8), 0, 0, -1, 0)
        for key, v in zip(KEYS, want):
            assert np.array_equal(r[key][q], v), (what, q, key, r[key][q], v)


def seeded_costs(rng, n, wide):
    return rng.integers(1, 1 << 32, n, dtype=np.uint64) if wide else rng.integers(1, 9, n).astype(np.uint64)


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for of the batch)
def test_oracle_on_every_route(vhp, oracle, monkeypatch, n):
    rng = np.random.default_rng(n + 211)
    cs = contexts(vhp, monkeypatch)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 10, 70 + m, 3, 14) for m in range(2)])
    sizes = [0, 1, 2, 3, 6] if n == 12 else [n // 3, 1, n // 3, 0, n - 2 * (n // 3) - 1]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = (np.arange(len(sizes)) % 2).astype(np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[mp], int(sx), int(sy)) for (sx, sy), mp in zip(srcs, pmap)])
    W = seeded_weights((len(sizes), ny, nx), rng)
    R = 20
    kmax = 6 if n == 12 else 10
    i = 0
    for sh in ("box", "disk"):
        for thr in (0.5, 0.0):
            base = problem_sets(fields, srcs, ptr, thr, R, sh == "disk")
            for vw in (None, seeded_views(vhp, rng, len(srcs), R)):
                psets = base if vw is None else \
                    [view_sets(s, srcs[a:b], vw[a:b], R, sh) for s, a, b in zip(base, ptr[:-1], ptr[1:])]
                for m in (1, 2, 3):
                    i += 1
                    w = W if i % 2 else None
                    wide = i % 3 == 0
                    cost = seeded_costs(rng, len(srcs), wide)
                    unit = 1 << 31 if wide else 4
                    budget = np.array([0, unit, 3 * unit, 12 * unit, U64_MAX][:len(sizes)], np.uint64)
                    quota = None if i % 4 else np.array([5, 0, 10**9, 300, 40][:len(sizes)], np.uint64)
                    for c in cs:
                        r = c.visibility_cover_budget_batch(occ, srcs, ptr, cost, budget, thr, R, shape_of(vhp, sh),
                                                            quota=quota, m=m, weights=w, views=vw, kmax=kmax,
                                                            group_map=gmap)
                        check(r, psets, ptr, kmax, m, cost, budget, quota, w, (ny, nx),
                              (n, sh, thr, vw is None, m, w is None, wide))
    for c in cs:
        c.close()


@pytest.mark.parametrize("n", [12, 400, 2500])
def test_unit_cost_identities(vhp, monkeypatch, n):
    """all costs 1: budget B and no quota is the view (m-fold) call with k = min(B, kmax), single its first pick; budget
    UINT64_MAX and a quota is the quota call, total included"""
    rng = np.random.default_rng(n + 223)
    cs = contexts(vhp, monkeypatch)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 10, 90 + m, 3, 14) for m in range(2)])
    sizes = [0, 1, 2, 3, 6] if n == 12 else [n // 3, 1, n // 3, 0, n - 2 * (n // 3) - 1]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = (np.arange(len(sizes)) % 2).astype(np.int32)
    W = seeded_weights((len(sizes), ny, nx), rng)
    R, kmax = 20, 9
    ones = np.ones(len(srcs), np.uint32)
    for sh in ("box", "disk"):
        for thr in (0.5, 0.0):
            for vw in (None, seeded_views(vhp, rng, len(srcs), R)):
                for m, w in ((1, None), (2, W), (3, None)):
                    for c in cs:
                        for B in (0, 1, 4, kmax + 3):
                            ref = reference(c, occ, srcs, vw, ptr, min(B, kmax), m, thr, R, shape_of(vhp, sh), w,
                                            gmap)
                            r = c.visibility_cover_budget_batch(occ, srcs, ptr, ones, B, thr, R, shape_of(vhp, sh),
                                                                m=m, weights=w, views=vw, kmax=kmax, group_map=gmap)
                            k = min(B, kmax)
                            for key in ("pick", "gain"):
                                assert np.array_equal(r[key][:, :k], ref[key]), (n, sh, thr, m, B, key)
                                assert (r[key][:, k:] == (-1 if key == "pick" else 0)).all()
                            assert np.array_equal(r["npicked"], ref["npicked"]) and np.array_equal(r["count"],
                                                                                                   ref["count"])
                            assert np.array_equal(r["spent"], r["npicked"].astype(np.uint64))
                            first = reference(c, occ, srcs, vw, ptr, 1, m, thr, R, shape_of(vhp, sh), w, gmap)
                            want_single = first["pick"][:, 0] if B >= 1 else np.full(len(sizes), -1, np.int32)
                            assert np.array_equal(r["single"], want_single), (n, sh, thr, m, B)
                            assert np.array_equal(r["single_gain"], first["gain"][:, 0] if B >= 1 else
                                                  np.zeros(len(sizes), np.uint64))
                        full = reference(c, occ, srcs, vw, ptr, kmax, m, thr, R, shape_of(vhp, sh), w, gmap)
                        tot = full["gain"].sum(1, dtype=np.uint64)
                        quota = np.array([0, 1, tot[2] // 2, tot[3] + 1, tot[4]][:len(sizes)], np.uint64)
                        qr = c.visibility_cover_quota_batch(occ, srcs, ptr, thr, R, shape_of(vhp, sh), quota=quota,
                                                            m=m, weights=w, views=vw, kmax=kmax, group_map=gmap)
                        r = c.visibility_cover_budget_batch(occ, srcs, ptr, ones, U64_MAX, thr, R, shape_of(vhp, sh),
                                                            quota=quota, m=m, weights=w, views=vw, kmax=kmax,
                                                            group_map=gmap)
                        for key in ("pick", "gain", "npicked", "count", "total", "reached"):
                            assert np.array_equal(r[key], qr[key]), (n, sh, thr, m, key)
    for c in cs:
        c.close()


def farey_costs(g1, g2, sign):
    """c1, c2 near 2^31 with g1 c2 - g2 c1 = sign (g1, g2 coprime)"""
    inv = pow(g1, -1, g2) if g2 > 1 else 0
    c2 = (sign * inv) % g2 if g2 > 1 else 1
    c2 += ((1 << 31) - c2) // g2 * g2
    c1 = (g1 * c2 - sign) // g2
    assert g1 * c2 - g2 * c1 == sign and 1 <= c1 < 1 << 32 and 1 <= c2 < 1 << 32
    return c1, c2


def test_farey_near_ties(ctx, vhp):
    """two candidates of gains near 2^30 with costs near 2^31 and g1 c2 - g2 c1 = +-1: their ratios differ by less than
    2^-60 of their size, below what fp64 resolves.  The exact winner is picked, and exactly equal ratios go to the
    smaller index"""
    rng = np.random.default_rng(227)
    nx = ny = 3000
    occ = rect_map(nx, ny, 20, 5, 3, 30)[None]
    srcs = np.stack([rng.integers(1000, 2000, 16), rng.integers(1000, 2000, 16)], 1).astype(np.int32)
    W = rng.integers(200, 256, (1, ny, nx), dtype=np.uint8)
    R = 1400
    # round-0 gains from singleton problems
    one = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, np.arange(len(srcs) + 1), 1, 1, 0.5, R, vhp.RANGE_DISK,
                                                  weights=np.repeat(W, len(srcs), 0))
    g = [int(v) for v in one["gain"][:, 0]]
    assert min(g) > 1 << 29
    pairs = [(i, j) for i in range(len(srcs)) for j in range(i + 1, len(srcs))
             if math.gcd(g[i], g[j]) == 1 and 0.6 < g[i] / g[j] < 1.6][:16]
    assert len(pairs) >= 8
    fp_blind = checked = 0
    for i, j in pairs:
        for sign in (1, -1):
            c1, c2 = farey_costs(g[i], g[j], sign)  # sign 1: g_i / c1 > g_j / c2 by 1 / (c1 c2)
            fp_blind += (g[i] / c1 > g[j] / c2) != (sign == 1) or g[i] / c1 == g[j] / c2
            for order in ((i, j), (j, i)):
                cost = np.array([c1, c2] if order == (i, j) else [c2, c1], np.uint32)
                r = ctx.visibility_cover_budget_batch(occ, srcs[list(order)], [0, 2], cost, U64_MAX, 0.5, R,
                                                      vhp.RANGE_DISK, weights=W, kmax=1)
                winner = i if sign == 1 else j
                assert int(r["pick"][0, 0]) == order.index(winner), (i, j, sign, order, c1, c2)
                assert int(r["gain"][0, 0]) == g[winner]
                checked += 1
        # exact tie: cost = g * t with the same t; the smaller index wins in both orders
        t = ((1 << 32) - 1) // max(g[i], g[j])
        for order in ((i, j), (j, i)):
            cost = np.array([g[order[0]] * t, g[order[1]] * t], np.uint32)
            r = ctx.visibility_cover_budget_batch(occ, srcs[list(order)], [0, 2], cost, U64_MAX, 0.5, R,
                                                  vhp.RANGE_DISK, weights=W, kmax=1)
            assert int(r["pick"][0, 0]) == 0, (i, j, order)
    assert checked >= 32 and fp_blind >= len(pairs)  # an fp64 ratio would get at least half of them wrong


def test_mixed_stopping_equals_each_problem_alone(ctx, vhp):
    rng = np.random.default_rng(229)
    nx, ny = 150, 110
    occ = np.stack([rect_map(nx, ny, 30, 50 + m, 3, 16) for m in range(2)])
    sizes = [30, 7, 0, 45, 12, 30, 1, 60, 25, 9, 40, 18]
    srcs, ptr = make_groups(rng, nx, ny, occ[0], sizes)
    gmap = (np.arange(len(sizes)) % 2).astype(np.int32)
    W = seeded_weights((len(sizes), ny, nx), rng)
    views = seeded_views(vhp, rng, len(srcs), 25)
    cost = rng.integers(1, 9, len(srcs)).astype(np.uint32)
    # budget (small), exhausted (no budget), kmax (kmax 5 below what the budget allows), quota
    budget = np.array([6, U64_MAX, 50, 4, U64_MAX, 10, 3, U64_MAX, 20, 1, U64_MAX, 7], np.uint64)
    quota = np.array([U64_MAX, U64_MAX, 0, U64_MAX, 900, U64_MAX, U64_MAX, 2000, U64_MAX, U64_MAX, 5000, U64_MAX],
                     np.uint64)
    for vw, m, kmax in ((None, 1, 60), (views, 2, 60), (views, 1, 5)):
        r = ctx.visibility_cover_budget_batch(occ, srcs, ptr, cost, budget, 0.5, 25, vhp.RANGE_DISK, quota=quota, m=m,
                                              weights=W, views=vw, kmax=kmax, group_map=gmap)
        for q in range(len(sizes)):
            a, b = ptr[q], ptr[q + 1]
            one = ctx.visibility_cover_budget_batch(occ, srcs[a:b], [0, b - a], cost[a:b], budget[q], 0.5, 25,
                                                    vhp.RANGE_DISK, quota=quota[q:q + 1], m=m, weights=W[q:q + 1],
                                                    views=None if vw is None else vw[a:b], kmax=kmax,
                                                    group_map=gmap[q:q + 1])
            for key in KEYS + ("reached", "best_single"):
                assert np.array_equal(r[key][q], one[key][0]), (q, key)
        assert (r["spent"] <= budget).all()
        assert r["reached"].any() and not r["reached"].all()
        assert (r["npicked"] == kmax).any() or kmax > 10


def test_a_loop_of_thousands_of_rounds(ctx, vhp):
    """one problem of 4000 candidates of range 2 on a 400^2 map with equal costs and a budget above their sum: the
    loop runs thousands of rounds, each the m-fold call's"""
    rng = np.random.default_rng(233)
    nx = ny = 400
    occ = rect_map(nx, ny, 200, 9, 3, 12)[None]
    srcs = np.stack([rng.integers(0, nx, 4000), rng.integers(0, ny, 4000)], 1).astype(np.int32)
    ptr = np.array([0, len(srcs)], np.int64)
    for m, w in ((1, None), (2, seeded_weights((1, ny, nx), rng))):
        u = ctx.visibility_cover_greedy_mfold_batch(occ, srcs, ptr, len(srcs), m, 0.5, 2, vhp.RANGE_BOX, weights=w)
        cost = np.full(len(srcs), 7, np.uint32)
        r = ctx.visibility_cover_budget_batch(occ, srcs, ptr, cost, 7 * 5000, 0.5, 2, vhp.RANGE_BOX, m=m, weights=w)
        assert r["npicked"][0] > 1000
        for key in ("pick", "gain", "npicked", "count"):
            assert np.array_equal(r[key], u[key]), (m, key)
        assert int(r["spent"][0]) == 7 * int(r["npicked"][0])
        # a budget that runs out part way: the first 1234 picks
        r = ctx.visibility_cover_budget_batch(occ, srcs, ptr, cost, 7 * 1234 + 6, 0.5, 2, vhp.RANGE_BOX, m=m,
                                              weights=w)
        assert r["npicked"][0] == 1234 and np.array_equal(r["pick"][0, :1234], u["pick"][0, :1234])


@pytest.mark.parametrize("mode,thr,views", [(1, 0.5, False), (1, 0.0, False), (1, 0.5, True), (2, 0.5, False)])
def test_launches_do_not_depend_on_costs_budgets_or_rounds(vhp, ctx, mode, thr, views):
    import torch
    nsrc, R = 40, 16
    occ_t = dev_maps(torch, 1, 600, 600, 7)
    xy = torch.from_numpy(sources(nsrc, 600, 600, 8)).cuda()
    vw = torch.from_numpy(vhp.sensor_views(np.arange(nsrc) * 70.0, 90, R)).cuda() if views else None
    gptr = torch.tensor([0, nsrc], dtype=torch.int64, device="cuda:0")
    pk = torch.empty((1, nsrc), dtype=torch.int32, device="cuda:0")
    cnt = torch.empty((1, 600, 600), dtype=torch.uint8, device="cuda:0")
    sg = torch.empty((1,), dtype=torch.int32, device="cuda:0")
    rng = np.random.default_rng(239)
    ctx.set_grid_sweep(mode)
    try:
        ctx.prepare_maps_dev(occ_t)
        counts = set()
        for costs, budget, quota, kmax in (((1, 2), 0, None, 5), ((1, 9), 30, None, 5), ((1, 1 << 32), U64_MAX, 300, 30),
                                           ((1, 2), U64_MAX, None, 1), ((5, 6), 4, 0, nsrc)):
            c_t = torch.from_numpy(rng.integers(*costs, nsrc).astype(np.uint32).view(np.int32)).cuda()
            b_t = torch.from_numpy(np.array([budget], np.uint64).view(np.int64)).cuda()
            q_t = None if quota is None else torch.from_numpy(np.array([quota], np.uint64).view(np.int64)).cuda()
            fn = lambda: ctx.visibility_cover_budget_batch_dev(occ_t, xy, gptr, c_t, b_t, kmax, thr, R,  # noqa: E731
                                                               vhp.RANGE_DISK, quota_t=q_t, m=2, pick_t=pk,
                                                               count_t=cnt, single_t=sg, views_t=vw)
            counts.add(launches_of(ctx, fn))
        assert len(counts) == 1, counts
        # the quota call's launches plus the output kernel
        q1 = torch.from_numpy(np.array([U64_MAX], np.uint64).view(np.int64)).cuda()
        ref = lambda: ctx.visibility_cover_quota_batch_dev(occ_t, xy, gptr, q1, 5, thr, R,  # noqa: E731
                                                           vhp.RANGE_DISK, m=2, pick_t=pk, count_t=cnt, views_t=vw)
        assert counts == {launches_of(ctx, ref) + 1}
    finally:
        ctx.set_grid_sweep(1)


def test_graph_is_fresh_after_the_buffers_grow(vhp):
    """a call, a larger call that grows the cover buffers, the first again, interleaved with the quota call: every
    result is unchanged"""
    c = vhp.Context(0)
    rng = np.random.default_rng(241)
    small = (np.stack([rect_map(80, 60, 8, 1, 3, 10)]), 80, 60, [6, 9, 4])
    big = (np.stack([rect_map(300, 250, 60, 2, 3, 20)]), 300, 250, [200, 150, 120, 90])
    runs = []
    for occ, nx, ny, sizes in (small, big):
        srcs, ptr = make_groups(rng, nx, ny, occ[0], sizes)
        W = seeded_weights((len(sizes), ny, nx), rng)
        runs.append((occ, srcs, ptr, W, seeded_views(vhp, rng, len(srcs), 18),
                     rng.integers(1, 9, len(srcs)).astype(np.uint32)))

    def budget_call(i):
        occ, srcs, ptr, W, vw, cost = runs[i]
        return c.visibility_cover_budget_batch(occ, srcs, ptr, cost, 30, 0.5, 18, vhp.RANGE_DISK, m=2, weights=W,
                                               views=vw)

    def quota_call(i):
        occ, srcs, ptr, W, vw, cost = runs[i]
        return c.visibility_cover_quota_batch(occ, srcs, ptr, 0.5, 18, vhp.RANGE_DISK, fraction=0.6, m=2, weights=W,
                                              views=vw)

    a0, o0 = budget_call(0), quota_call(0)
    b0 = budget_call(1)
    quota_call(1)
    a1 = budget_call(0)
    b1 = budget_call(1)
    o2 = quota_call(0)
    a2 = budget_call(0)
    for x, y in ((a0, a1), (a0, a2), (b0, b1), (o0, o2)):
        for key in x:
            assert np.array_equal(x[key], y[key]), key
    assert a0["npicked"].any() and b0["npicked"].any()
    c.close()


def test_dev_equals_host(vhp):
    import torch
    rng = np.random.default_rng(251)
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
    for R, sh, thr, kmax, m, views, wide in ((5, "disk", 0.5, 7, 2, True, False), (33, "box", 0.0, 40, 3, False, True),
                                             (60, "disk", 1e-9, 50, 1, True, True)):
        vw = seeded_views(vhp, rng, len(srcs), R) if views else None
        v_t = torch.from_numpy(vw).cuda() if views else None
        cost = seeded_costs(rng, len(srcs), wide).astype(np.uint32)
        unit = 1 << 30 if wide else 3
        budget = np.array([0, unit, 5 * unit, U64_MAX, 2 * unit, 9 * unit, 40 * unit], np.uint64)
        for w, quota in ((None, None), (W, np.array([10, 0, 5, 10**6, 300, 1, 2000], np.uint64))):
            host = c.visibility_cover_budget_batch(occ, srcs, ptr, cost, budget, thr, R, shape_of(vhp, sh),
                                                   quota=quota, m=m, weights=w, views=vw, kmax=kmax, group_map=gmap)
            with torch.cuda.stream(stream):
                c_t = torch.from_numpy(cost.view(np.int32)).cuda()
                b_t = torch.from_numpy(budget.view(np.int64)).cuda()
                q_t = None if quota is None else torch.from_numpy(quota.view(np.int64)).cuda()
                outs = dict(pick=torch.full((ng, kmax), 5, dtype=torch.int32, device="cuda:0"),
                            gain=torch.full((ng, kmax), 5, dtype=torch.int64, device="cuda:0"),
                            npicked=torch.full((ng,), 5, dtype=torch.int32, device="cuda:0"),
                            count=torch.full((ng, ny, nx), 5, dtype=torch.uint8, device="cuda:0"),
                            total=torch.full((ng,), 5, dtype=torch.int64, device="cuda:0"),
                            spent=torch.full((ng,), 5, dtype=torch.int64, device="cuda:0"),
                            single=torch.full((ng,), 5, dtype=torch.int32, device="cuda:0"),
                            single_gain=torch.full((ng,), 5, dtype=torch.int64, device="cuda:0"))
                c.visibility_cover_budget_batch_dev(occ_t, xy_t, ptr_t, c_t, b_t, kmax, thr, R, shape_of(vhp, sh),
                                                    quota_t=q_t, m=m, group_map_t=gm_t,
                                                    weights_t=None if w is None else w_t, views_t=v_t,
                                                    **{k + "_t": v for k, v in outs.items()})
            c.synchronize()
            for key, t in outs.items():
                got = t.cpu().numpy()
                if got.dtype == np.int64:
                    got = got.view(np.uint64)
                assert np.array_equal(got, host[key]), (R, sh, thr, key)
    c.close()


def test_two_4gb_runs_equal_one_problem_at_a_time(ctx, vhp):
    """8 weighted problems on 12000^2 maps with count: about 0.6 GB of device memory each, so the host form runs them
    in two runs, each with its slice of costs and budgets"""
    nx = ny = 12000
    rng = np.random.default_rng(257)
    occ = np.stack([rect_map(nx, ny, 3000, 200 + m, 10, 80) for m in range(2)]).astype(np.uint8)
    sizes = [5, 1, 9, 3, 6, 2, 7, 4]
    xy = np.stack([rng.integers(0, nx, sum(sizes)), rng.integers(0, ny, sum(sizes))], 1).astype(np.int32)
    xy[:3] = [(0, 0), (nx - 1, ny - 1), (6000, 0)]
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    gmap = (np.arange(8) % 2).astype(np.int32)
    W = rng.integers(0, 256, (8, ny, nx), dtype=np.uint8)
    R = 48
    views = seeded_views(vhp, rng, len(xy), R)
    cost = rng.integers(1, 9, len(xy)).astype(np.uint32)
    budget = np.array([0, 3, 8, 100, U64_MAX, 12, 5, 9], np.uint64)
    quota = np.array([U64_MAX, 1, 5000, 10**6, U64_MAX, 20000, 300000, 2], np.uint64)
    r = ctx.visibility_cover_budget_batch(occ, xy, ptr, cost, budget, 0.5, R, vhp.RANGE_DISK, quota=quota, m=2,
                                          weights=W, views=views, kmax=6, group_map=gmap)
    for q in range(8):
        a, b = ptr[q], ptr[q + 1]
        one = ctx.visibility_cover_budget_batch(occ, xy[a:b], [0, b - a], cost[a:b], budget[q], 0.5, R,
                                                vhp.RANGE_DISK, quota=quota[q:q + 1], m=2, weights=W[q:q + 1],
                                                views=views[a:b], kmax=6, group_map=gmap[q:q + 1])
        for key in KEYS + ("reached", "best_single"):
            assert np.array_equal(r[key][q], one[key][0]), (q, key)
    assert r["npicked"][0] == 0 and (r["npicked"][2:] > 0).all()


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    good = np.array([(4, 1, 0, 0, 1), (4, 1, 1, 1, 1), (0, -1, 0, 1, 0)], np.int32)
    cost = np.array([2, 3, 1], np.uint32)
    bad = [
        dict(radius=-1), dict(radius=16384), dict(shape=2), dict(kmax=-1), dict(m=0), dict(m=256),
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32)),  # candidate outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                 # map out of range
        dict(group_ptr=[1, 3]),                                      # does not start at 0
        dict(threshold=float("nan")),
        dict(views=np.array([good[0], (5, 1, 0, 0, 1), good[2]], np.int32)),
        dict(cost=np.array([2, 0, 1], np.uint32)),
    ]
    for b in bad:
        kw = dict(src_xy=srcs, group_ptr=[0, 3], cost=cost, budget=10, threshold=0.5, radius=4, shape=vhp.RANGE_DISK,
                  views=good, kmax=2, m=2)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_budget_batch(occ, kw.pop("src_xy"), kw.pop("group_ptr"), kw.pop("cost"),
                                            kw.pop("budget"), kw.pop("threshold"), kw.pop("radius"), kw.pop("shape"),
                                            **kw)
        assert e.value.status == -1, b
        if "kmax" in b:
            assert b"vhp_visibility_cover_budget_batch: kmax < 0" in c.lib.vhp_last_error(c.h)
        if "cost" in b:
            assert b"the cost of candidate 1 is 0" in c.lib.vhp_last_error(c.h)
        r = c.visibility_cover_budget_batch(occ, srcs, [0, 3], cost, 10, 0.5, 4, vhp.RANGE_DISK, views=good, kmax=2,
                                            m=2)
        assert r["npicked"][0] == 2  # still works
    # a zero cost is reported before any candidate is read: it wins over a candidate outside the grid
    with pytest.raises(vhp.VhpError):
        c.visibility_cover_budget_batch(occ, np.array([(1, 1), (30, 5), (7, 2)], np.int32), [0, 3], [1, 0, 1], 10, 0.5,
                                        4, vhp.RANGE_DISK, kmax=2)
    assert b"cost of candidate 1 is 0" in c.lib.vhp_last_error(c.h)
    occ_u8 = np.ones((1, 20, 30), np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    npk = np.zeros(1, np.int32)
    one = vhp.CoverBudgetOut(None, None, npk.ctypes.data, None, None, None, None, None)
    single = np.zeros(1, np.int32)
    only_single = vhp.CoverBudgetOut(None, None, None, None, None, None, single.ctypes.data, None)
    gp = np.array([0, 3], np.int64)
    bud = np.array([10], np.uint64)
    fn = c.lib.vhp_visibility_cover_budget_batch
    args = lambda xy, views, ptr, cst, b, out: (c.h, vp(occ_u8), 1, 30, 20, vp(xy), views, vp(ptr), None, 1, 2, 4,  # noqa: E731,E501
                                                 vhp.RANGE_BOX, 0.5, None, 2, None, cst, b, C.byref(out))
    assert fn(*args(srcs, None, gp, None, vp(bud), one)) == -1 and b"cost is NULL" in c.lib.vhp_last_error(c.h)
    assert fn(*args(srcs, None, gp, vp(cost), None, one)) == -1 and b"budget is NULL" in c.lib.vhp_last_error(c.h)
    none = vhp.CoverBudgetOut(None, None, None, None, None, None, None, None)
    assert fn(*args(srcs, None, gp, vp(cost), vp(bud), none)) == -1 and b"no output" in c.lib.vhp_last_error(c.h)
    assert fn(*args(srcs, None, gp, vp(cost), vp(bud), only_single)) == 0 and single[0] >= 0  # single alone
    big = np.array([0, 2**28], np.int64)
    assert fn(*args(srcs, vp(good), big, vp(cost), vp(bud), one)) == -1 and b"2^28" in c.lib.vhp_last_error(c.h)
    # no problem needs no budget, no candidate no cost
    empty = np.array([0], np.int64)
    assert fn(c.h, vp(occ_u8), 1, 30, 20, vp(srcs), None, vp(empty), None, 0, 2, 4, vhp.RANGE_BOX, 0.5, None, 2, None,
              None, None, C.byref(one)) == 0
    # kmax 0: no pick, single -1
    r = c.visibility_cover_budget_batch(occ, srcs, [0, 3], cost, 10, 0.5, 4, vhp.RANGE_DISK, kmax=0)
    assert r["single"].tolist() == [-1] and r["spent"].tolist() == [0] and r["total"].tolist() == [0]
    assert not r["count"].any() and r["pick"].shape == (1, 0)
    # the _dev form: bad arguments at once, a zero cost through the device error flag (bit 5)
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    pk = torch.empty((2, 3), dtype=torch.int32, device=d)
    xy_ok = torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d)
    ptr_ok = torch.tensor([0, 1, 3], dtype=torch.int64, device=d)
    c_t = torch.tensor([1, 2, 3], dtype=torch.int32, device=d)
    b_t = torch.tensor([100, 100], dtype=torch.int64, device=d)
    for radius, kmax, m, cst, bd in ((-1, 3, 2, c_t, b_t), (4, -1, 2, c_t, b_t), (4, 3, 0, c_t, b_t),
                                     (4, 3, 2, None, b_t), (4, 3, 2, c_t, None)):
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_cover_budget_batch_dev(occ_t, xy_ok, ptr_ok, cst, bd, kmax, 0.5, radius, vhp.RANGE_BOX, m=m,
                                                pick_t=pk)
        assert e.value.status == -1
    c.synchronize()
    sg = torch.empty((2,), dtype=torch.int32, device=d)
    for zero_at in (0, 1, 2):
        zc = torch.tensor([0 if i == zero_at else 1 for i in range(3)], dtype=torch.int32, device=d)
        c.visibility_cover_budget_batch_dev(occ_t, xy_ok, ptr_ok, zc, b_t, 3, 0.5, 4, vhp.RANGE_BOX, m=2, pick_t=pk,
                                            single_t=sg)
        with pytest.raises(vhp.VhpError) as e:
            c.synchronize()
        assert e.value.status == -1 and b"cost is 0" in c.lib.vhp_last_error(c.h), zero_at
        # that candidate is never picked nor the singleton
        q, local = (0, 0) if zero_at == 0 else (1, zero_at - 1)
        assert local not in pk[q].tolist() and int(sg[q]) != local, zero_at
        c.visibility_cover_budget_batch_dev(occ_t, xy_ok, ptr_ok, c_t, b_t, 3, 0.5, 4, vhp.RANGE_BOX, m=2, pick_t=pk)
        c.synchronize()
    # problem 0: (1, 1) alone; problem 1: (3, 1) of cost 2 sees 7 x 5 written cells, (2, 2) of cost 3 sees 6 x 6: the
    # ratio picks (3, 1) first (35 / 2 > 36 / 3), the best singleton is (2, 2)
    gn = torch.empty((2, 3), dtype=torch.int64, device=d)
    sp = torch.empty((2,), dtype=torch.int64, device=d)
    c.visibility_cover_budget_batch_dev(occ_t, xy_ok, ptr_ok, c_t, b_t, 3, 0.5, 4, vhp.RANGE_BOX, m=2, pick_t=pk,
                                        gain_t=gn, spent_t=sp, single_t=sg)
    c.synchronize()
    assert pk.tolist() == [[0, -1, -1], [0, 1, -1]] and sg.tolist() == [0, 1] and sp.tolist() == [1, 5]
    assert gn[1, 0] == 35
    c.close()
