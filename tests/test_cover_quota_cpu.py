"""The definition of quota sensor placement (vhp_visibility_cover_quota_batch), pinned on the CPU oracle with the numpy
m-fold greedy of test_cover_mfold_cpu: each problem runs the m-fold greedy and stops at the first pick after which the
summed gain reaches its quota, at a gain of 0, or at kmax picks; the result is a prefix of the greedy with k = kmax.
Also the Python helper that turns a fraction into quotas."""
import itertools

import numpy as np
import pytest

from test_cover_cpu import sets_of
from test_cover_mfold_cpu import mgreedy
from test_cover_weighted_cpu import seeded_weights
from test_merge_range_cpu import seeded_groups

U64_MAX = np.iinfo(np.uint64).max


def qgreedy(sets, kmax, m, quota, weights=None):
    """pick, gain, npicked, count, total of the quota greedy: the m-fold greedy, stopped once sum of gain >= quota"""
    pick = np.full(kmax, -1, np.int32)
    gain = np.zeros(kmax, np.uint64)
    shape = sets[0].shape if sets else (1, 1)
    W = np.ones(shape, np.int64) if weights is None else weights.astype(np.int64)
    cnt = np.zeros(shape, np.int64)
    taken = np.zeros(len(sets), bool)
    total = n = 0
    while total < quota and n < min(kmax, len(sets)):
        gains = [0 if taken[i] else int(W[S & (cnt < m)].sum()) for i, S in enumerate(sets)]
        p = int(np.argmax(gains))
        if gains[p] == 0:
            break
        pick[n], gain[n] = p, gains[p]
        total += gains[p]
        n += 1
        taken[p] = True
        cnt[sets[p]] = np.minimum(cnt[sets[p]] + 1, m)
    return pick, gain, n, cnt.astype(np.uint8), total


def prefix_of(sets, kmax, m, quota, weights=None):
    """the prefix rule: the m-fold greedy of kmax rounds, cut at the first j with sum of gain[:j] >= quota, and the
    count of the greedy run with k = that j"""
    pick, gain, n, _ = mgreedy(sets, kmax, m, weights)
    sums = np.concatenate([[0], np.cumsum(gain[:n].astype(object))])
    j = next((i for i, s in enumerate(sums) if s >= quota), n)
    pick[j:], gain[j:] = -1, 0
    _, _, _, cnt = mgreedy(sets, j, m, weights)
    return pick, gain, j, cnt, int(sums[j])


def cases(oracle, seed):
    rng = np.random.default_rng(seed)
    for occ, srcs, R in seeded_groups():
        for thr, disk in ((0.5, True), (0.0, False)):
            sets = sets_of(oracle, occ, srcs, thr, R, disk)
            for W in (None, seeded_weights(occ.shape, rng)):
                yield sets, W


def test_the_quota_greedy_is_the_prefix_rule(oracle):
    for sets, W in cases(oracle, 61):
        for m in (1, 2, 3):
            _, gain, n, _ = mgreedy(sets, len(sets), m, W)
            full = int(gain.sum())
            for quota in (0, 1, full // 3, full // 2, full - 1, full, full + 1, U64_MAX):
                for kmax in (0, 1, 3, len(sets), len(sets) + 2):
                    got = qgreedy(sets, kmax, m, quota, W)
                    want = prefix_of(sets, kmax, m, quota, W)
                    for a, b in zip(got, want):
                        assert np.array_equal(a, b), (m, quota, kmax)


def test_quota_0_makes_no_pick(oracle):
    for sets, W in cases(oracle, 67):
        pick, gain, n, cnt, total = qgreedy(sets, 4, 2, 0, W)
        assert n == 0 and total == 0 and (pick == -1).all() and not gain.any() and not cnt.any()


def test_a_quota_equal_to_a_prefix_sum_stops_at_that_pick(oracle):
    for sets, W in cases(oracle, 71):
        for m in (1, 2):
            _, gain, n, _ = mgreedy(sets, len(sets), m, W)
            sums = np.cumsum(gain[:n].astype(np.int64))
            for j in range(n):
                assert qgreedy(sets, len(sets), m, int(sums[j]), W)[2] == j + 1
                # one more unit needs the next pick (or, after the last positive gain, is never reached)
                assert qgreedy(sets, len(sets), m, int(sums[j]) + 1, W)[2] == min(j + 2, n)


def test_an_unreachable_quota_stops_at_gain_0(oracle):
    for sets, W in cases(oracle, 73):
        for m in (1, 3):
            pick, gain, n, _ = mgreedy(sets, len(sets) + 1, m, W)
            full = int(gain.sum())
            got = qgreedy(sets, len(sets) + 1, m, full + 1, W)
            assert got[2] == n and got[4] == full and got[4] < full + 1  # not reached
            assert np.array_equal(got[0], pick) and np.array_equal(got[1], gain)
            assert got[2] < len(sets) + 1


def test_kmax_caps_the_picks(oracle):
    for sets, W in cases(oracle, 79):
        _, gain, n, _ = mgreedy(sets, len(sets), 2, W)
        for kmax in range(n):
            got = qgreedy(sets, kmax, 2, U64_MAX, W)
            assert got[2] == kmax and got[4] == int(gain[:kmax].sum())


def test_fraction_is_the_documented_ceil():
    import visibility_heuristic_path_planner_b200 as vhp
    rng = np.random.default_rng(83)
    W = seeded_weights((3, 7, 9), rng)
    for p in (0.0, 0.25, 0.5, 0.9, 0.95, 1.0, 1.5, 1 / 3):
        for m in (1, 2, 3):
            got = vhp._cover_quota(None, p, m, W, 3, (7, 9))
            want = [int(np.ceil(p * m * float(W[q].astype(np.int64).sum()))) for q in range(3)]
            assert got.dtype == np.uint64 and got.tolist() == want, (p, m)
            assert vhp._cover_quota(None, p, m, None, 2, (7, 9)).tolist() == [int(np.ceil(p * m * 63.0))] * 2
    assert vhp._cover_quota(None, None, 1, None, 2, (7, 9)).tolist() == [U64_MAX] * 2
    assert vhp._cover_quota(5, None, 1, None, 3, (7, 9)).tolist() == [5] * 3
    assert vhp._cover_quota([0, U64_MAX], None, 1, None, 2, (7, 9)).tolist() == [0, U64_MAX]
    for bad in (dict(quota=1, fraction=0.5), dict(fraction=-0.1), dict(fraction=float("nan")), dict(quota=-1),
                dict(quota=[1.5, 2.0])):
        with pytest.raises(ValueError):
            vhp._cover_quota(bad.get("quota"), bad.get("fraction"), 1, None, 2, (7, 9))


def harmonic(n):
    return sum(1.0 / i for i in range(1, n + 1))


def test_full_cover_is_within_h_of_the_optimum(oracle):
    """quota UINT64_MAX, kmax = the group's size, unweighted, m = 1: greedy set cover of the union, within H(max |S|)
    of the fewest candidates that cover it (brute force)"""
    rng = np.random.default_rng(89)
    cases_run = 0
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        extra = [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(4)]
        cand = np.concatenate([srcs, np.array(extra, np.int32).reshape(-1, 2)])[:10]
        sets = sets_of(oracle, occ, cand, 0.5, max(1, R // 3), True)
        union = np.any(sets, axis=0)
        _, _, n, cnt, total = qgreedy(sets, len(sets), 1, U64_MAX)
        assert np.array_equal(cnt.astype(bool), union) and total == int(union.sum())
        opt = next(k for k in range(len(sets) + 1)
                   if any(np.array_equal(np.any([sets[i] for i in c], axis=0) if c else np.zeros_like(union), union)
                          for c in itertools.combinations(range(len(sets)), k)))
        assert n <= harmonic(max(int(S.sum()) for S in sets)) * opt, (occ.shape, n, opt)
        assert n >= opt
        cases_run += 1
    assert cases_run > 0
