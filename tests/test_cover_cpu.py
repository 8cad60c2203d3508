"""The definition of greedy sensor placement (vhp_visibility_cover_greedy_batch), pinned on the CPU oracle with a numpy
greedy reference: candidate c covers S(c), the cells where it would add 1 to vhp_visibility_merge_range_batch's count
(in range, not on its never-written border, fp64 value >= threshold); each round picks the candidate that adds the
most cells of the target to the union, ties to the smallest index, and stops at a gain of 0."""
import itertools

import numpy as np

from test_merge_cpu import writes_mask
from test_merge_range_cpu import fold_range, range_mask, seeded_groups

THRS = (0.5, 1e-9, 0.0, -1.0)


def cover_set(field, sx, sy, thr, R, disk):
    """S(c) of a candidate at (sx, sy) from its full fp64 field"""
    ny, nx = field.shape
    return range_mask(nx, ny, sx, sy, R, disk) & writes_mask(nx, ny, sx, sy) & (field >= thr)


def greedy(sets, k, target=None):
    """pick, gain, npicked, covered (bool) of the greedy over the candidate sets (list of bool (ny, nx))"""
    shape = sets[0].shape if sets else (1, 1)
    T = np.ones(shape, bool) if target is None else target
    U = np.zeros(shape, bool)
    pick = np.full(k, -1, np.int32)
    gain = np.zeros(k, np.uint32)
    n = 0
    for r in range(min(k, len(sets))):
        gains = [int((S & T & ~U).sum()) for S in sets]
        p = int(np.argmax(gains))  # the first maximum: ties to the smallest index
        if gains[p] == 0:
            break
        pick[r], gain[r], n = p, gains[p], r + 1
        U |= sets[p]
    return pick, gain, n, U


def sets_of(oracle, occ, srcs, thr, R, disk):
    return [cover_set(oracle.compute_visibility(occ, int(sx), int(sy)), int(sx), int(sy), thr, R, disk)
            for sx, sy in srcs]


def seeded_targets(shape, rng):
    return rng.random(shape) < 0.6


def test_cover_set_is_the_range_merge_count(oracle):
    for occ, srcs, R in seeded_groups():
        for sx, sy in srcs:
            f = oracle.compute_visibility(occ, int(sx), int(sy))
            for thr in THRS:
                for disk in (False, True):
                    want = fold_range([f], [(sx, sy)], thr, occ.shape, R, disk)[2] > 0
                    assert np.array_equal(cover_set(f, int(sx), int(sy), thr, R, disk), want), (occ.shape, R, thr)


def test_gains_sum_to_the_covered_target_and_do_not_increase(oracle):
    rng = np.random.default_rng(7)
    for occ, srcs, R in seeded_groups():
        for thr, disk in ((0.5, True), (0.0, False)):
            sets = sets_of(oracle, occ, srcs, thr, R, disk)
            for target in (None, seeded_targets(occ.shape, rng)):
                pick, gain, n, U = greedy(sets, 4, target)
                T = np.ones(occ.shape, bool) if target is None else target
                assert int(gain.sum()) == int((U & T).sum())
                assert (np.diff(gain.astype(np.int64)) <= 0).all()
                assert (pick[n:] == -1).all() and (gain[n:] == 0).all() and (gain[:n] > 0).all()
                want = np.zeros(occ.shape, bool)
                for p in pick[:n]:
                    want |= sets[p]
                assert np.array_equal(U, want)


def test_within_one_minus_one_over_e_of_the_optimum(oracle):
    rng = np.random.default_rng(11)
    bound = 1.0 - 1.0 / np.e
    cases = 0
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        extra = [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(4)]
        cand = np.concatenate([srcs, np.array(extra, np.int32).reshape(-1, 2)])[:10]
        sets = sets_of(oracle, occ, cand, 0.5, max(1, R // 3), True)
        for k in (1, 2, 3):
            _, gain, _, _ = greedy(sets, k)
            opt = max(int(np.logical_or.reduce([sets[i] for i in c]).sum())
                      for c in itertools.combinations(range(len(sets)), k))
            assert int(gain.sum()) >= bound * opt, (occ.shape, k)
            cases += 1
    assert cases == 180


def test_more_picks_are_a_second_call_on_the_complement(oracle):
    """k1 + k2 picks = k1 picks, then k2 picks whose target is the complement of what the first ones cover"""
    rng = np.random.default_rng(5)
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        more = [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(6)]
        cand = np.concatenate([srcs, np.array(more, np.int32)])
        sets = sets_of(oracle, occ, cand, 0.5, R, False)
        for k1, k2 in ((1, 2), (2, 3), (3, 1)):
            pick, gain, n, U = greedy(sets, k1 + k2)
            p1, g1, n1, U1 = greedy(sets, k1)
            p2, g2, n2, U2 = greedy(sets, k2, ~U1)
            assert np.array_equal(pick, np.concatenate([p1, p2]))  # (a first call that stops leaves nothing)
            assert np.array_equal(gain, np.concatenate([g1, g2]))
            assert np.array_equal(U, U1 | U2) and n == n1 + n2


def test_ties_duplicates_and_occupied_candidates(oracle):
    occ = np.ones((20, 30))
    occ[5, 7] = 0
    # two disjoint boxes of the same size: the smaller index wins the tie, whatever the order
    cand = [(20, 10), (5, 10), (20, 10), (7, 5)]
    sets = sets_of(oracle, occ, cand, 0.5, 2, False)
    assert sets[0].sum() == sets[1].sum() == 25
    pick, gain, n, U = greedy(sets, 4)
    assert list(pick) == [0, 1, -1, -1] and list(gain) == [25, 25, 0, 0] and n == 2
    # the duplicate of a pick has gain 0 from then on, so it never is picked; an occupied candidate covers nothing
    assert not sets[3].any()
    pick, gain, n, _ = greedy([sets[2], sets[0], sets[3]], 3)
    assert list(pick) == [0, -1, -1] and n == 1
    # at threshold <= 0 every cell in range that the sweep writes counts, occupied candidate included
    assert sets_of(oracle, occ, [(7, 5)], 0.0, 2, False)[0].sum() == 25
