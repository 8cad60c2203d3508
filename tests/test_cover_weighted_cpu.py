"""The definition of weighted greedy sensor placement (vhp_visibility_cover_greedy_weighted_batch), pinned on the CPU
oracle with a numpy weighted greedy: S(c) is the coverage set of vhp_visibility_cover_greedy_batch (test_cover_cpu);
each round picks the candidate whose cells not yet covered have the largest summed uint8 weight, ties to the smallest
index, and stops at a gain of 0."""
import itertools

import numpy as np

from test_cover_cpu import greedy, sets_of
from test_merge_range_cpu import seeded_groups


def wgreedy(sets, k, weights=None):
    """pick, gain (uint64), npicked, covered (bool) of the weighted greedy over the candidate sets (list of bool
    (ny, nx)); weights uint8 (ny, nx), None: every cell weighs 1"""
    shape = sets[0].shape if sets else (1, 1)
    W = np.ones(shape, np.uint64) if weights is None else weights.astype(np.uint64)
    U = np.zeros(shape, bool)
    pick = np.full(k, -1, np.int32)
    gain = np.zeros(k, np.uint64)
    n = 0
    for r in range(min(k, len(sets))):
        gains = [int(W[S & ~U].sum()) for S in sets]
        p = int(np.argmax(gains))  # the first maximum: ties to the smallest index
        if gains[p] == 0:
            break
        pick[r], gain[r], n = p, gains[p], r + 1
        U |= sets[p]
    return pick, gain, n, U


def seeded_weights(shape, rng):
    """uint8 weights with zeros and 255 in them"""
    w = rng.integers(0, 256, shape).astype(np.uint8)
    w[rng.random(shape) < 0.2] = 0
    w[rng.random(shape) < 0.05] = 255
    return w


def test_gains_sum_to_the_covered_weight_and_do_not_increase(oracle):
    rng = np.random.default_rng(17)
    for occ, srcs, R in seeded_groups():
        for thr, disk in ((0.5, True), (0.0, False)):
            sets = sets_of(oracle, occ, srcs, thr, R, disk)
            for W in (None, seeded_weights(occ.shape, rng)):
                pick, gain, n, U = wgreedy(sets, 4, W)
                Wf = np.ones(occ.shape, np.uint64) if W is None else W.astype(np.uint64)
                assert int(gain.sum()) == int(Wf[U].sum())
                assert (np.diff(gain.astype(np.int64)) <= 0).all()
                assert (pick[n:] == -1).all() and (gain[n:] == 0).all() and (gain[:n] > 0).all()
                want = np.zeros(occ.shape, bool)
                for p in pick[:n]:
                    want |= sets[p]
                assert np.array_equal(U, want)


def test_within_one_minus_one_over_e_of_the_optimum(oracle):
    rng = np.random.default_rng(19)
    bound = 1.0 - 1.0 / np.e
    cases = 0
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        extra = [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(4)]
        cand = np.concatenate([srcs, np.array(extra, np.int32).reshape(-1, 2)])[:10]
        sets = sets_of(oracle, occ, cand, 0.5, max(1, R // 3), True)
        W = seeded_weights(occ.shape, rng).astype(np.int64)
        for k in (1, 2, 3):
            _, gain, _, _ = wgreedy(sets, k, W.astype(np.uint8))
            opt = max(int(W[np.logical_or.reduce([sets[i] for i in c])].sum())
                      for c in itertools.combinations(range(len(sets)), k))
            assert int(gain.sum()) >= bound * opt, (occ.shape, k)
            cases += 1
    assert cases == 180


def test_binary_weights_are_the_target(oracle):
    """weights in {0, 1} give vhp_visibility_cover_greedy_batch's greedy with that target, and no weights its greedy
    without one"""
    rng = np.random.default_rng(23)
    for occ, srcs, R in seeded_groups():
        sets = sets_of(oracle, occ, srcs, 0.5, R, False)
        T = rng.random(occ.shape) < 0.6
        for k in (1, 3, 8):
            for w, t in ((T.astype(np.uint8), T), (None, None)):
                pw, gw, nw, Uw = wgreedy(sets, k, w)
                pick, gain, n, U = greedy(sets, k, t)
                assert np.array_equal(pw, pick) and np.array_equal(gw, gain.astype(np.uint64))
                assert nw == n and np.array_equal(Uw, U)


def test_constant_weights_scale_the_gains(oracle):
    for occ, srcs, R in seeded_groups():
        sets = sets_of(oracle, occ, srcs, 0.5, R, True)
        pick, gain, n, U = greedy(sets, 5)
        for c in (1, 7, 255):
            pw, gw, nw, Uw = wgreedy(sets, 5, np.full(occ.shape, c, np.uint8))
            assert np.array_equal(pw, pick) and np.array_equal(gw, gain.astype(np.uint64) * c)
            assert nw == n and np.array_equal(Uw, U)


def test_ties_zero_weights_duplicates_and_occupied_candidates(oracle):
    occ = np.ones((20, 30))
    occ[5, 7] = 0
    cand = [(20, 10), (5, 10), (20, 10), (7, 5), (12, 3)]
    sets = sets_of(oracle, occ, cand, 0.5, 2, False)
    W = np.ones((20, 30), np.uint8)
    # equal weight sums on disjoint boxes: the smaller index wins the tie
    pick, gain, n, _ = wgreedy(sets, 5, W)
    assert list(pick[:2]) == [0, 1] and list(gain[:2]) == [25, 25]
    # a heavy cell decides over a larger count of light ones
    W2 = W.copy()
    W2[10, 5] = 200
    pick, gain, n, _ = wgreedy(sets, 1, W2)
    assert list(pick) == [1] and list(gain) == [224]
    # zero weights: a candidate that only covers zero-weight cells has gain 0 and is never picked, though the cells
    # it would cover are in the union where another pick covers them
    W3 = W.copy()
    W3[8:13, 18:23] = 0  # the box of candidates 0 and 2
    pick, gain, n, U = wgreedy(sets, 5, W3)
    assert 0 not in pick[:n] and 2 not in pick[:n] and not U[8:13, 18:23].any()
    pick, gain, n, U = wgreedy(sets[:2], 5, W3)
    assert list(pick) == [1, -1, -1, -1, -1] and n == 1
    # the duplicate of a pick has gain 0 from then on; an occupied candidate covers nothing
    assert not sets[3].any()
    pick, gain, n, _ = wgreedy([sets[2], sets[0], sets[3]], 3, seeded_weights((20, 30), np.random.default_rng(1)))
    assert list(pick) == [0, -1, -1] and n == 1
    # all weights 0: nothing is picked
    pick, gain, n, U = wgreedy(sets, 3, np.zeros((20, 30), np.uint8))
    assert n == 0 and not U.any() and (pick == -1).all()
