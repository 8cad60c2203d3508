"""The definition of directional greedy sensor placement (vhp_visibility_cover_greedy_view_batch), pinned on the CPU
oracle: each candidate's coverage set is S(c) of vhp_visibility_cover_greedy_batch (test_cover_cpu) narrowed to its
view (r, a, b), which view_mask tests cell by cell; the greedy is the m-fold greedy of test_cover_mfold_cpu on those
sets.  Also sensor_views, the helper that turns headings and fields of view into integer vectors."""
import itertools

import numpy as np
import pytest

from test_cover_cpu import sets_of
from test_cover_mfold_cpu import f_of, mgreedy
from test_cover_weighted_cpu import seeded_weights
from test_merge_range_cpu import seeded_groups


def view_mask(dx, dy, view, R, shape):
    """bool mask of the cells (dx, dy) (int arrays, relative to the sensor) in the view (r, ax, ay, bx, by); shape
    "box" or "disk".  Every cell is tested directly: range, then the direction rule of include/vhp.h."""
    r, ax, ay, bx, by = (int(v) for v in view)
    assert 0 <= r <= R and (ax, ay) != (0, 0) and (bx, by) != (0, 0)
    dx, dy = np.asarray(dx, np.int64), np.asarray(dy, np.int64)
    rng = (np.abs(dx) <= r) & (np.abs(dy) <= r) if shape == "box" else dx * dx + dy * dy <= r * r
    c1 = ax * dy - ay * dx  # cross(a, d)
    c2 = dx * by - dy * bx  # cross(d, b)
    cab, dab = ax * by - ay * bx, ax * bx + ay * by
    if cab > 0:
        direction = (c1 >= 0) & (c2 >= 0)
    elif cab < 0 or dab < 0:
        direction = (c1 >= 0) | (c2 >= 0)
    else:
        direction = np.ones(dx.shape, bool)
    return rng & (direction | ((dx == 0) & (dy == 0)))


def view_sets(sets, srcs, views, R, shape):
    """S_view(c) = S(c) & view(c) of every candidate"""
    out = []
    for S, (sx, sy), v in zip(sets, srcs, views):
        Y, X = np.indices(S.shape)
        out.append(S & view_mask(X - int(sx), Y - int(sy), v, R, shape))
    return out


def random_views(rng, n, R):
    """views with random integer vectors, among them axis-aligned, opposite, equal and non-primitive ones"""
    out = []
    for i in range(n):
        a = [int(t) for t in rng.integers(-5, 6, 2)]
        if a == [0, 0]:
            a = [1, 0]
        kind = i % 5
        b = ([-a[0], -a[1]] if kind == 0 else list(a) if kind == 1 else [2 * a[0], 2 * a[1]] if kind == 2 else
             [int(t) for t in rng.integers(-5, 6, 2)])
        if b == [0, 0]:
            b = [0, 1]
        out.append([int(rng.integers(0, R + 1))] + a + b)
    return np.array(out, np.int32)


def test_omnidirectional_views_are_the_mfold_greedy(oracle):
    rng = np.random.default_rng(61)
    for occ, srcs, R in seeded_groups():
        for thr, shape in ((0.5, "disk"), (0.0, "box")):
            sets = sets_of(oracle, occ, srcs, thr, R, shape == "disk")
            omni = [(R, 3, -7, 3, -7), (R, 1, 0, 2, 0), (R, -32767, 5, -32767, 5)] * 3
            vs = view_sets(sets, srcs, omni[:len(srcs)], R, shape)
            assert all(np.array_equal(a, b) for a, b in zip(vs, sets))
            W = seeded_weights(occ.shape, rng)
            for m in (1, 2):
                for a, b in zip(mgreedy(vs, 5, m, W), mgreedy(sets, 5, m, W)):
                    assert np.array_equal(a, b)


def test_opposite_vectors_give_the_closed_half_plane():
    Y, X = np.indices((41, 41))
    dx, dy = X - 20, Y - 20
    for a in ((1, 0), (0, 1), (3, -2), (-7, 5), (32767, 1), (2, 4)):
        ax, ay = a
        half = view_mask(dx, dy, (20, ax, ay, -ax, -ay), 20, "box")
        assert np.array_equal(half, ax * dy - ay * dx >= 0)
        other = view_mask(dx, dy, (20, -ax, -ay, ax, ay), 20, "box")
        assert (half | other).all()
        assert np.array_equal(half & other, ax * dy - ay * dx == 0)  # the line through the sensor
        assert half[20, 20] and other[20, 20]


def test_nested_sectors_and_radii_give_nested_sets():
    Y, X = np.indices((61, 61))
    dx, dy = X - 30, Y - 30
    for shape in ("box", "disk"):
        for h in range(0, 360, 23):
            prev = None
            for fov in (1, 30, 90, 179, 180, 181, 270, 359, 360):
                v = [int(t) for t in np.rint(1000 * np.array([np.cos(np.radians(h - fov / 2)),
                                                               np.sin(np.radians(h - fov / 2)),
                                                               np.cos(np.radians(h + fov / 2)),
                                                               np.sin(np.radians(h + fov / 2))]))]
                if fov == 360:
                    v[2:] = v[:2]
                cur = view_mask(dx, dy, [30] + v, 30, shape)
                if prev is not None:
                    assert not (prev & ~cur).any(), (shape, h, fov)
                prev = cur
            assert prev.sum() == ((np.abs(dx) <= 30) & (np.abs(dy) <= 30) if shape == "box"
                                  else dx * dx + dy * dy <= 900).sum()
        for view in ((1, 0, 1, 1), (3, 1, -1, -2), (1, 1, 1, 1)):
            prev = None
            for r in range(31):
                cur = view_mask(dx, dy, (r,) + view, 30, shape)
                if prev is not None:
                    assert not (prev & ~cur).any(), (shape, view, r)
                prev = cur


def test_sensor_cell_is_in_its_view(oracle):
    rng = np.random.default_rng(67)
    for occ, srcs, R in seeded_groups():
        sets = sets_of(oracle, occ, srcs, 0.5, R, True)
        views = random_views(rng, len(srcs), R)
        for S, (sx, sy), V in zip(sets, srcs, view_sets(sets, srcs, views, R, "disk")):
            assert V[sy, sx] == S[sy, sx]
            assert not (V & ~S).any()


def test_within_one_minus_one_over_e_of_the_optimum(oracle):
    rng = np.random.default_rng(71)
    bound = 1.0 - 1.0 / np.e
    cases = 0
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        extra = [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(4)]
        cand = np.concatenate([srcs, np.array(extra, np.int32).reshape(-1, 2)])[:10]
        Rc = max(1, R // 3)
        sets = view_sets(sets_of(oracle, occ, cand, 0.5, Rc, True), cand, random_views(rng, len(cand), Rc), Rc,
                         "disk")
        W = seeded_weights(occ.shape, rng)
        for m in (1, 2):
            for k in (2, 3):
                _, gain, _, _ = mgreedy(sets, k, m, W)
                opt = max(f_of(sets, list(c), m, W) for c in itertools.combinations(range(len(sets)), k))
                assert int(gain.sum()) >= bound * opt, (occ.shape, m, k)
                cases += 1
    assert cases == 240


def test_sensor_views():
    from visibility_heuristic_path_planner_b200 import sensor_views
    v = sensor_views([0, 45, 200], 360, 7)
    assert v.dtype == np.int32 and v.shape == (3, 5)
    assert (v[:, 0] == 7).all() and np.array_equal(v[:, 1:3], v[:, 3:5])
    assert v[0, 1:].tolist() == [32767, 0, 32767, 0]
    Y, X = np.indices((41, 41))
    dx, dy = X - 20, Y - 20
    for h in (0, 30, 90, 135, 217, 300):
        v = sensor_views(h, 90, 20)[0]
        mask = view_mask(dx, dy, v, 20, "disk")
        for t in (-40, -20, 0, 20, 40):  # interior directions of the 90 degree view
            u = np.radians(h + t)
            assert mask[20 + int(round(15 * np.sin(u))), 20 + int(round(15 * np.cos(u)))], (h, t)
        u = np.radians(h + 180)
        assert not mask[20 + int(round(15 * np.sin(u))), 20 + int(round(15 * np.cos(u)))], h
    # the +x axis, heading 90 (towards +y, the next rows): a = (32767, 0) rotated by 45 degrees either side
    v = sensor_views(90, 90, 3)[0]
    assert v.tolist() == [3, 23170, 23170, -23170, 23170]
    assert sensor_views([10, 20], [60, 300], [4, 5]).shape == (2, 5)
    for fov in (1e-4, 0.001):
        with pytest.raises(ValueError):
            sensor_views(33, fov, 5)
    for fov in (0, -10):
        with pytest.raises(ValueError):
            sensor_views(0, fov, 5)


def test_new_symbols_are_exported():
    import visibility_heuristic_path_planner_b200 as vhp
    lib = vhp.load_library()
    for name in ("vhp_visibility_cover_greedy_view_batch", "vhp_visibility_cover_greedy_view_batch_dev"):
        assert hasattr(lib, name)
