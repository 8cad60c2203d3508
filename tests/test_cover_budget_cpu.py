"""The definition of budgeted sensor placement (vhp_visibility_cover_budget_batch), pinned on the CPU oracle with a numpy
greedy built on the m-fold greedy's conventions: each problem picks, among the candidates not yet picked whose cost fits
what is left of its budget and whose gain is positive, the one of largest gain / cost (exact rational comparison, ties
to the smallest index), until none is eligible, kmax picks are made or the quota is reached.  Also the identities with
the fixed-k and quota greedies, the approximation bound against brute force, the 128-bit ratio key against Fraction
(and where a 64-bit fixed point or an fp64 ratio fails), and the Python handling of cost and budget."""
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest

from test_cover_cpu import sets_of
from test_cover_mfold_cpu import f_of, mgreedy
from test_cover_quota_cpu import qgreedy
from test_cover_view_cpu import random_views, view_sets
from test_cover_weighted_cpu import seeded_weights
from test_merge_range_cpu import seeded_groups

U64_MAX = np.iinfo(np.uint64).max
IDX_BITS = 28


def bgreedy(sets, kmax, m, cost, budget, quota=None, weights=None):
    """pick, gain, npicked, count, total, spent, single, single_gain of the budget greedy"""
    pick = np.full(kmax, -1, np.int32)
    gain = np.zeros(kmax, np.uint64)
    shape = sets[0].shape if sets else (1, 1)
    W = np.ones(shape, np.int64) if weights is None else weights.astype(np.int64)
    cnt = np.zeros(shape, np.int64)
    taken = np.zeros(len(sets), bool)
    g0 = [int(W[S].sum()) for S in sets]
    fits0 = [i for i in range(len(sets)) if g0[i] > 0 and int(cost[i]) <= budget]
    single = max(fits0, key=lambda i: (g0[i], -i)) if kmax > 0 and fits0 else -1
    single_gain = g0[single] if single >= 0 else 0
    total = spent = n = 0
    while n < min(kmax, len(sets)) and (quota is None or total < quota):
        best = None
        for i, S in enumerate(sets):
            g = 0 if taken[i] else int(W[S & (cnt < m)].sum())
            if g > 0 and int(cost[i]) <= budget - spent:
                # exact: g / c > bg / bc  <=>  g * bc > bg * c; ties keep the smaller index (the first found)
                if best is None or g * int(cost[best[0]]) > best[1] * int(cost[i]):
                    best = (i, g)
        if best is None:
            break
        p, g = best
        pick[n], gain[n] = p, g
        total += g
        spent += int(cost[p])
        n += 1
        taken[p] = True
        cnt[sets[p]] = np.minimum(cnt[sets[p]] + 1, m)
    return pick, gain, n, cnt.astype(np.uint8), total, spent, single, single_gain


def ratio_key(g, c, k):
    """the 128-bit key of kernels_cover.cu, as the kernel computes it: g / c, then two 32-bit long-division steps"""
    hi, r0 = divmod(g, c)
    d1, r1 = divmod(r0 << 32, c)
    d2 = (r1 << 32) // c
    f = (hi << 64) | (d1 << 32) | d2
    assert f == (g << 64) // c
    return (f << IDX_BITS) | ((1 << IDX_BITS) - 1 - k)


def cases(oracle, seed, views=False):
    rng = np.random.default_rng(seed)
    for occ, srcs, R in seeded_groups():
        for thr, disk in ((0.5, True), (0.0, False)):
            sets = sets_of(oracle, occ, srcs, thr, R, disk)
            if views:
                sets = view_sets(sets, srcs, random_views(rng, len(srcs), R), R, "disk" if disk else "box")
            for W in (None, seeded_weights(occ.shape, rng)):
                yield sets, W, rng


def test_unit_costs_are_the_fixed_k_greedy(oracle):
    """identity 1: all costs 1, no quota, budget B is the m-fold (or view) greedy with k = min(B, kmax)"""
    for views in (False, True):
        for sets, W, rng in cases(oracle, 101 + views, views):
            ones = np.ones(len(sets), np.int64)
            for m in (1, 2, 3):
                for B, kmax in ((0, 4), (1, 4), (3, 4), (4, 3), (len(sets) + 1, len(sets))):
                    pick, gain, n, cnt, total, spent, single, sg = bgreedy(sets, kmax, m, ones, B, None, W)
                    want = mgreedy(sets, min(B, kmax), m, W)
                    assert np.array_equal(pick[:min(B, kmax)], want[0]) and (pick[min(B, kmax):] == -1).all()
                    assert np.array_equal(gain[:min(B, kmax)], want[1]) and n == want[2]
                    assert np.array_equal(cnt, want[3]) and spent == n and total == int(want[1].sum())
                    first = mgreedy(sets, 1, m, W)
                    assert single == (int(first[0][0]) if B >= 1 and kmax >= 1 else -1)
                    assert sg == (int(first[1][0]) if single >= 0 else 0)


def test_unit_costs_without_a_budget_are_the_quota_greedy(oracle):
    """identity 2: all costs 1, budget UINT64_MAX, a quota: the quota greedy with the same quota and kmax"""
    for sets, W, rng in cases(oracle, 103):
        ones = np.ones(len(sets), np.int64)
        for m in (1, 2):
            full = int(mgreedy(sets, len(sets), m, W)[1].sum())
            for quota in (0, 1, full // 2, full, full + 1):
                for kmax in (0, 2, len(sets)):
                    got = bgreedy(sets, kmax, m, ones, int(U64_MAX), quota, W)
                    want = qgreedy(sets, kmax, m, quota, W)
                    for a, b in zip(got[:5], want):
                        assert np.array_equal(a, b), (m, quota, kmax)


def test_scaling_costs_and_budget_changes_nothing(oracle):
    """identity 3: costs * s and budget * s give the same pick, gain and npicked"""
    for sets, W, rng in cases(oracle, 107):
        cost = rng.integers(1, 9, len(sets))
        for B in (3, 10, 40):
            base = bgreedy(sets, len(sets), 2, cost, B, None, W)
            for s in (2, 7, 1 << 20):
                got = bgreedy(sets, len(sets), 2, cost * s, B * s, None, W)
                for a, b in zip(got[:3], base[:3]):
                    assert np.array_equal(a, b), (B, s)
                assert got[5] == base[5] * s and got[6] == base[6]


def test_every_cost_above_the_budget_picks_nothing(oracle):
    """identity 4"""
    for sets, W, rng in cases(oracle, 109):
        cost = rng.integers(6, 20, len(sets))
        pick, gain, n, cnt, total, spent, single, sg = bgreedy(sets, 5, 2, cost, 5, None, W)
        assert n == 0 and total == 0 and spent == 0 and single == -1 and sg == 0
        assert (pick == -1).all() and not gain.any() and not cnt.any()


def test_budget_is_respected_and_every_pick_was_affordable(oracle):
    for sets, W, rng in cases(oracle, 113):
        cost = rng.integers(1, 9, len(sets))
        for B in (1, 5, 13, 40):
            pick, gain, n, _, total, spent, _, _ = bgreedy(sets, len(sets), 2, cost, B, None, W)
            left = B
            for p in pick[:n]:
                assert int(cost[p]) <= left
                left -= int(cost[p])
            assert spent == B - left <= B and total == int(gain.sum())
            assert len(set(pick[:n].tolist())) == n and (gain[:n] > 0).all()
            # stopped because nothing else fits with a positive gain
            if n < len(sets):
                chosen = list(pick[:n])
                Wf = np.ones(sets[0].shape, np.uint8) if W is None else W
                base = f_of(sets, chosen, 2, Wf)
                assert all(int(cost[i]) > left or f_of(sets, chosen + [i], 2, Wf) == base
                           for i in range(len(sets)) if i not in chosen)


def test_ratios_are_exact_and_ties_go_to_the_smallest_index():
    """two candidates of gains 3 and 2 with costs 3 and 2 tie at ratio 1: the smaller index wins; with cost 2 and 3
    the ratios 3/2 and 2/3 are ordered by value, not by gain"""
    S = np.zeros((3, 5), bool)
    a, b = S.copy(), S.copy()
    a[0, :3] = True
    b[2, :2] = True
    assert bgreedy([a, b], 1, 1, [3, 2], 10)[0][0] == 0
    assert bgreedy([b, a], 1, 1, [2, 3], 10)[0][0] == 0
    c = S.copy()
    c[1, :4] = True  # gain 4 at cost 3 beats gain 3 at cost 3 and gain 2 at cost 2
    assert bgreedy([a, b, c], 1, 1, [3, 2, 3], 10)[0][0] == 2
    assert bgreedy([a, b, c], 1, 1, [3, 1, 3], 10)[0][0] == 1  # 2 / 1 beats 4 / 3


def test_occupied_and_zero_gain_candidates_are_never_picked(oracle):
    for occ, srcs, R in seeded_groups():
        wall = np.argwhere(occ == 0)
        if len(wall) == 0:
            continue
        cand = np.concatenate([srcs, wall[:3, ::-1].astype(np.int32)])
        sets = sets_of(oracle, occ, cand, 0.5, R, True)
        cost = np.ones(len(cand), np.int64)  # cheapest possible: still never picked
        pick, gain, n, *_ = bgreedy(sets, len(cand), 1, cost, len(cand))
        assert not set(pick[:n].tolist()) & set(range(len(srcs), len(cand)))
        assert (gain[:n] > 0).all()


def test_best_of_greedy_and_single_is_within_the_bound_of_the_optimum():
    """max(total, single_gain) >= (1 - 1/e) / 2 * OPT for m = 1, 2, and >= (1 - 1/sqrt(e)) * OPT for m = 1, on a few
    hundred tiny random instances against brute force"""
    rng = np.random.default_rng(127)
    runs = 0
    for t in range(300):
        ny, nx, n = 3, 4, int(rng.integers(3, 8))
        sets = [rng.random((ny, nx)) < rng.uniform(0.15, 0.6) for _ in range(n)]
        W = rng.integers(0, 6, (ny, nx)).astype(np.uint8)
        cost = rng.integers(1, 9, n)
        B = int(rng.integers(1, 16))
        for m in (1, 2):
            _, _, _, _, total, spent, single, sg = bgreedy(sets, n, m, cost, B, None, W)
            assert spent <= B
            opt = max(f_of(sets, list(c), m, W) for r in range(n + 1) for c in itertools.combinations(range(n), r)
                      if sum(int(cost[i]) for i in c) <= B)
            best = max(total, sg)
            assert best <= opt
            assert best >= (1 - 1 / math.e) / 2 * opt - 1e-9, (t, m)
            if m == 1:
                assert best >= (1 - 1 / math.sqrt(math.e)) * opt - 1e-9, t
            runs += 1
    assert runs == 600


def farey_pairs(rng, count):
    """pairs (g1, c1), (g2, c2) with g1 c2 - g2 c1 = +-1, g < 2^36, c < 2^32, c near 2^31 or spread: adjacent Farey
    fractions, whose ratios differ by 1 / (c1 c2)"""
    out = []
    while len(out) < count:
        c1 = int(rng.integers(1 << 30, (1 << 32) - 1)) if rng.random() < 0.5 else int(rng.integers(2, 1 << 32))
        g1 = int(rng.integers(1, 1 << 36))
        if math.gcd(g1, c1) != 1:
            continue
        # g1 * c2 - g2 * c1 = 1: c2 = g1^-1 mod c1 (then g2 = (g1 c2 - 1) / c1)
        c2 = pow(g1, -1, c1)
        g2 = (g1 * c2 - 1) // c1
        if not (1 <= c2 < (1 << 32) and 1 <= g2 < (1 << 36)):
            continue
        out.append(((g1, c1), (g2, c2)) if rng.random() < 0.5 else ((g2, c2), (g1, c1)))
    return out


def test_ratio_key_orders_like_fraction():
    rng = np.random.default_rng(131)
    pairs = [((int(rng.integers(1, 1 << 36)), int(rng.integers(1, 1 << 32))),
              (int(rng.integers(1, 1 << 36)), int(rng.integers(1, 1 << 32)))) for _ in range(20000)]
    pairs += [((int(rng.integers(1, 64)), int(rng.integers(1, 9))), (int(rng.integers(1, 64)), int(rng.integers(1, 9))))
              for _ in range(5000)]
    for _ in range(2000):  # exact ties: (g, c) and (s g, s c)
        g, c = int(rng.integers(1, 1 << 20)), int(rng.integers(1, 1 << 16))
        s = int(rng.integers(1, 1 << 15))
        pairs.append(((g, c), (g * s, c * s)))
    pairs += farey_pairs(rng, 5000)
    pairs += [((1, 1), (1, 1)), (((1 << 36) - 1, 1), ((1 << 36) - 2, 1)), ((1, (1 << 32) - 1), (1, (1 << 32) - 2))]
    ties = 0
    for (g1, c1), (g2, c2) in pairs:
        k1, k2 = int(rng.integers(0, 1 << 27)), int(rng.integers(0, 1 << 27))
        if k1 == k2:
            k2 += 1
        a, b = ratio_key(g1, c1, k1), ratio_key(g2, c2, k2)
        assert a < 1 << 128 and b < 1 << 128 and a > 0
        fa, fb = Fraction(g1, c1), Fraction(g2, c2)
        if fa != fb:
            assert (a > b) == (fa > fb), ((g1, c1), (g2, c2))
        else:
            ties += 1
            assert (a > b) == (k1 < k2)
    assert ties > 2000
    assert ratio_key(1, (1 << 32) - 1, (1 << 28) - 1) > 1 << 32  # positive gain: never the empty slot's 0


def test_fixed_point_and_fp64_ratios_fail_on_farey_neighbours():
    """the near-ties the exact key is built for: a 64-bit fixed point floor(g 2^32 / c) and an fp64 g / c both call
    some of them equal (or order them wrongly), the 128-bit key orders every one"""
    rng = np.random.default_rng(137)
    fixed_bad = fp_bad = 0
    for (g1, c1), (g2, c2) in farey_pairs(rng, 2000):
        want = Fraction(g1, c1) > Fraction(g2, c2)
        assert (ratio_key(g1, c1, 0) > ratio_key(g2, c2, 1)) == want
        f1, f2 = (g1 << 32) // c1, (g2 << 32) // c2
        fixed_bad += f1 == f2 or (f1 > f2) != want
        d1, d2 = g1 / c1, g2 / c2
        fp_bad += d1 == d2 or (d1 > d2) != want
    assert fixed_bad > 1000 and fp_bad > 100, (fixed_bad, fp_bad)


def test_cost_and_budget_arguments():
    import visibility_heuristic_path_planner_b200 as vhp
    assert vhp._cover_cost([1, 2, 3], 3).dtype == np.uint32
    assert vhp._cover_cost(np.array([1, 0xffffffff], np.int64), 2).tolist() == [1, 0xffffffff]
    assert vhp._cover_cost(np.array([5], np.uint32), 1).tolist() == [5]
    assert vhp._cover_cost(np.zeros(0, np.int64), 0).shape == (0,)
    assert vhp._cover_cost([0, 1], 2).tolist() == [0, 1]  # a zero is the library's error, with its index
    for bad, n in (([1, 2], 3), ([[1, 2]], 2), ([1.5, 2.0], 2), ([-1, 2], 2), ([1, 1 << 32], 2), (["a", 1], 2)):
        with pytest.raises(ValueError):
            vhp._cover_cost(bad, n)
    assert vhp._cover_u64(7, 3, "budget").tolist() == [7] * 3
    assert vhp._cover_u64([0, U64_MAX], 2, "budget").tolist() == [0, U64_MAX]
    assert vhp._cover_u64(np.array([3, 4], np.int32), 2, "budget").dtype == np.uint64
    for bad in (-1, [1.5, 2.0], [1, -2], "x"):
        with pytest.raises(ValueError, match="budget"):
            vhp._cover_u64(bad, 2, "budget")
    with pytest.raises(ValueError):
        vhp._cover_u64([1, 2, 3], 2, "budget")


def test_new_symbols_are_exported():
    import visibility_heuristic_path_planner_b200 as vhp
    lib = vhp.load_library(build_if_missing=False)
    assert lib.vhp_visibility_cover_budget_batch and lib.vhp_visibility_cover_budget_batch_dev
    assert [f for f, _ in vhp.CoverBudgetOut._fields_] == ["pick", "gain", "npicked", "count", "total", "spent",
                                                           "single", "single_gain"]
