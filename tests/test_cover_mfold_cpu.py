"""The definition of redundant (m-fold) greedy sensor placement (vhp_visibility_cover_greedy_mfold_batch), pinned on
the CPU oracle with a numpy m-fold greedy: S(c) is the coverage set of vhp_visibility_cover_greedy_batch
(test_cover_cpu); f(A) = sum of W(x) * min(cnt_A(x), m); each round picks the candidate, not yet picked, whose cells
covered fewer than m times have the largest summed uint8 weight, ties to the smallest index, and stops at a gain of 0."""
import itertools

import numpy as np

from test_cover_cpu import sets_of
from test_cover_weighted_cpu import seeded_weights, wgreedy
from test_merge_range_cpu import seeded_groups


def mgreedy(sets, k, m, weights=None):
    """pick, gain (uint64), npicked, count (uint8, min(m, picks covering the cell)) of the m-fold greedy over the
    candidate sets (list of bool (ny, nx)); weights uint8 (ny, nx), None: every cell weighs 1"""
    shape = sets[0].shape if sets else (1, 1)
    W = np.ones(shape, np.uint64) if weights is None else weights.astype(np.uint64)
    cnt = np.zeros(shape, np.int64)
    taken = np.zeros(len(sets), bool)
    pick = np.full(k, -1, np.int32)
    gain = np.zeros(k, np.uint64)
    n = 0
    for r in range(min(k, len(sets))):
        gains = [0 if taken[i] else int(W[S & (cnt < m)].sum()) for i, S in enumerate(sets)]
        p = int(np.argmax(gains))  # the first maximum: ties to the smallest index
        if gains[p] == 0:
            break
        pick[r], gain[r], n = p, gains[p], r + 1
        taken[p] = True
        cnt[sets[p]] = np.minimum(cnt[sets[p]] + 1, m)
    return pick, gain, n, cnt.astype(np.uint8)


def f_of(sets, chosen, m, W):
    """f of a set of candidate indices: sum of W * min(m, number of chosen sets covering the cell)"""
    c = np.sum([sets[i] for i in chosen], axis=0, dtype=np.int64) if chosen else 0
    return int((W.astype(np.int64) * np.minimum(c, m)).sum())


def test_m_1_is_the_weighted_greedy(oracle):
    rng = np.random.default_rng(41)
    for occ, srcs, R in seeded_groups():
        for thr, disk in ((0.5, True), (0.0, False)):
            sets = sets_of(oracle, occ, srcs, thr, R, disk)
            for W in (None, seeded_weights(occ.shape, rng)):
                for k in (1, 4, 8):
                    pick, gain, n, cnt = mgreedy(sets, k, 1, W)
                    pw, gw, nw, U = wgreedy(sets, k, W)
                    assert np.array_equal(pick, pw) and np.array_equal(gain, gw) and n == nw
                    assert np.array_equal(cnt, U.astype(np.uint8))


def test_gains_sum_to_f_do_not_increase_and_picks_are_distinct(oracle):
    rng = np.random.default_rng(43)
    for occ, srcs, R in seeded_groups():
        for thr, disk in ((0.5, True), (0.0, False)):
            sets = sets_of(oracle, occ, srcs, thr, R, disk)
            for W in (None, seeded_weights(occ.shape, rng)):
                Wf = np.ones(occ.shape, np.uint8) if W is None else W
                for m in (2, 3, 255):
                    pick, gain, n, cnt = mgreedy(sets, 6, m, W)
                    picks = [int(p) for p in pick[:n]]
                    assert len(set(picks)) == n
                    full = np.sum([sets[p] for p in picks], axis=0, dtype=np.int64) if n else np.zeros(occ.shape)
                    assert np.array_equal(cnt, np.minimum(full, m).astype(np.uint8))
                    assert int(gain.sum()) == f_of(sets, picks, m, Wf)
                    assert (np.diff(gain.astype(np.int64)) <= 0).all()
                    assert (pick[n:] == -1).all() and (gain[n:] == 0).all() and (gain[:n] > 0).all()


def test_identical_candidates_are_both_picked(oracle):
    """with m >= 2 a duplicate of a pick keeps its gain, so it can be the next argmax; with m = 1 it drops to 0"""
    occ = np.ones((20, 30))
    sets = sets_of(oracle, occ, [(20, 10), (20, 10), (5, 10)], 0.5, 2, False)
    assert sets[0].sum() == sets[2].sum() == 25
    for m in (2, 3):
        pick, gain, n, cnt = mgreedy(sets, 3, m)
        assert list(pick) == [0, 1, 2] and list(gain) == [25, 25, 25] and n == 3  # 1 wins the tie with 2
        assert cnt[8:13, 18:23].min() == 2 and cnt[8:13, 3:8].min() == 1
    pick, gain, n, _ = mgreedy(sets, 3, 1)
    assert list(pick) == [0, 2, -1] and n == 2
    # a heavier third candidate is taken before the duplicate, which comes after it
    W = np.ones((20, 30), np.uint8)
    W[10, 5] = 9
    pick, gain, n, _ = mgreedy(sets, 3, 2, W)
    assert list(pick) == [2, 0, 1] and list(gain) == [33, 25, 25]


def test_occupied_candidates_are_never_picked(oracle):
    occ = np.ones((20, 30))
    occ[5, 7] = 0
    sets = sets_of(oracle, occ, [(7, 5), (20, 10), (7, 5), (5, 12)], 0.5, 2, False)
    assert not sets[0].any() and not sets[2].any()
    for m in (1, 2, 5):
        pick, gain, n, _ = mgreedy(sets, 4, m)
        assert 0 not in pick[:n] and 2 not in pick[:n] and n == 2


def test_m_above_the_candidates_picks_every_positive_gain(oracle):
    """cnt never reaches m, so no gain ever drops: every candidate of positive weight is picked, heaviest first"""
    rng = np.random.default_rng(47)
    for occ, srcs, R in seeded_groups():
        sets = sets_of(oracle, occ, srcs, 0.5, R, True)
        W = seeded_weights(occ.shape, rng)
        w0 = [int(W[S].astype(np.int64).sum()) for S in sets]
        pick, gain, n, _ = mgreedy(sets, len(sets) + 2, len(sets) + 1, W)
        want = sorted((i for i in range(len(sets)) if w0[i] > 0), key=lambda i: (-w0[i], i))
        assert list(pick[:n]) == want and list(gain[:n]) == [w0[i] for i in want]


def test_within_one_minus_one_over_e_of_the_optimum(oracle):
    rng = np.random.default_rng(53)
    bound = 1.0 - 1.0 / np.e
    cases = 0
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        extra = [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(4)]
        cand = np.concatenate([srcs, np.array(extra, np.int32).reshape(-1, 2)])[:10]
        sets = sets_of(oracle, occ, cand, 0.5, max(1, R // 3), True)
        W = seeded_weights(occ.shape, rng)
        for m in (2, 3):
            for k in (2, 3, 4):
                _, gain, _, _ = mgreedy(sets, k, m, W)
                opt = max(f_of(sets, list(c), m, W) for c in itertools.combinations(range(len(sets)), k))
                assert int(gain.sum()) >= bound * opt, (occ.shape, m, k)
                cases += 1
    assert cases == 360
