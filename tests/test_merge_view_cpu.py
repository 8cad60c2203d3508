"""The definition of directional merged visibility (vhp_visibility_merge_view_batch), pinned on the CPU oracle: the
range merge of test_merge_range_cpu where source k only contributes to the cells of its view (r, a, b), which
view_mask of test_cover_view_cpu tests cell by cell.  vmax is the max of the fields masked to each view, and first /
count take the range merge's "writes" rule narrowed to the view."""
import numpy as np

from test_cover_view_cpu import random_views, view_mask
from test_merge_cpu import writes_mask
from test_merge_range_cpu import fields_of, fold_range, range_mask, seeded_groups


def fold_masked(fields, srcs, thr, masks):
    """vmax / first / count of one group from its full fp64 fields, source k contributing on masks[k] only"""
    ny, nx = fields[0].shape
    vmax = np.zeros((ny, nx))
    first = np.full((ny, nx), -1, np.int32)
    count = np.zeros((ny, nx), np.uint32)
    for k, (f, (sx, sy), m) in enumerate(zip(fields, srcs, masks)):
        vmax = np.maximum(vmax, np.where(m, f, 0.0))
        hit = m & (f >= thr) & writes_mask(nx, ny, int(sx), int(sy))
        first[(first < 0) & hit] = k
        count += hit
    return vmax, first, count


def view_masks(shape, srcs, views, R, sh):
    ny, nx = shape
    Y, X = np.indices((ny, nx))
    return [range_mask(nx, ny, int(sx), int(sy), R, sh == "disk") & view_mask(X - int(sx), Y - int(sy), v, R, sh)
            for (sx, sy), v in zip(srcs, views)]


def fold_view(fields, srcs, views, thr, R, sh):
    """vmax / first / count of one group of sources with views (shape sh: "box" or "disk")"""
    return fold_masked(fields, srcs, thr, view_masks(fields[0].shape, srcs, views, R, sh))


def ray_masks(shape, srcs, views):
    """the cells on the two boundary rays {t a, t b : t >= 0} of each source's sector"""
    ny, nx = shape
    Y, X = np.indices((ny, nx))
    out = []
    for (sx, sy), (_, ax, ay, bx, by) in zip(srcs, views):
        dx, dy = X - int(sx), Y - int(sy)
        ra = (ax * dy - ay * dx == 0) & (ax * dx + ay * dy >= 0)
        rb = (bx * dy - by * dx == 0) & (bx * dx + by * dy >= 0)
        out.append(ra | rb)
    return out


def cases():
    for occ, srcs, R in seeded_groups():
        for thr, sh in ((0.5, "disk"), (0.0, "box"), (1e-9, "disk")):
            yield occ, srcs, R, thr, sh


def test_omnidirectional_views_are_the_range_merge(oracle):
    for occ, srcs, R, thr, sh in cases():
        fields = fields_of(oracle, occ, srcs)
        omni = np.array([(R, 3, -7, 3, -7), (R, 1, 0, 2, 0), (R, -32767, 5, -32767, 5)] * 2, np.int32)[:len(srcs)]
        got = fold_view(fields, srcs, omni, thr, R, sh)
        want = fold_range(fields, srcs, thr, occ.shape, R, sh == "disk")
        for g, w in zip(got, want):
            assert np.array_equal(g, w)


def test_complementary_sectors_add_up_to_omni_plus_the_rays(oracle):
    """a -> b and b -> a cover every direction together and overlap on the two rays only"""
    rng = np.random.default_rng(71)
    for occ, srcs, R, thr, sh in cases():
        fields = fields_of(oracle, occ, srcs)
        ab = random_views(rng, len(srcs), R)
        ab[:, 0] = R
        for i, v in enumerate(ab):  # a and b must not point the same way
            ax, ay, bx, by = (int(t) for t in v[1:])
            if ax * by - ay * bx == 0 and ax * bx + ay * by > 0:
                ab[i, 3:] = (-ay, ax)
        ba = ab[:, [0, 3, 4, 1, 2]]
        rng_masks = [range_mask(occ.shape[1], occ.shape[0], int(sx), int(sy), R, sh == "disk") for sx, sy in srcs]
        omni = fold_masked(fields, srcs, thr, rng_masks)
        rays = fold_masked(fields, srcs, thr, [m & r for m, r in zip(rng_masks, ray_masks(occ.shape, srcs, ab))])
        v_ab = fold_view(fields, srcs, ab, thr, R, sh)
        v_ba = fold_view(fields, srcs, ba, thr, R, sh)
        assert np.array_equal(v_ab[2] + v_ba[2], omni[2] + rays[2])
        assert np.array_equal(np.maximum(v_ab[0], v_ba[0]), omni[0])


def test_nested_sectors_and_radii_nest(oracle):
    import visibility_heuristic_path_planner_b200 as vhp
    rng = np.random.default_rng(72)
    for occ, srcs, R, thr, sh in cases():
        fields = fields_of(oracle, occ, srcs)
        heading = rng.uniform(0, 360, len(srcs))
        prev = None
        for fov, r in ((40, R // 3), (90, R // 2), (90, R), (200, R), (360, R)):
            views = vhp.sensor_views(heading, fov, r)
            cur = fold_view(fields, srcs, views, thr, R, sh)
            if prev is not None:
                assert (prev[2] <= cur[2]).all() and (prev[0] <= cur[0]).all(), (fov, r)
            prev = cur


def test_zero_range_covers_the_source_cells_only(oracle):
    rng = np.random.default_rng(73)
    for occ, srcs, R, thr, sh in cases():
        fields = fields_of(oracle, occ, srcs)
        views = random_views(rng, len(srcs), R)
        views[:, 0] = 0
        vmax, first, count = fold_view(fields, srcs, views, thr, R, sh)
        want, want_vmax = np.zeros(occ.shape, np.uint32), np.zeros(occ.shape)
        want_first = np.full(occ.shape, -1, np.int32)
        for k, (f, (sx, sy)) in enumerate(zip(fields, srcs)):
            want_vmax[sy, sx] = max(want_vmax[sy, sx], f[sy, sx])
            if f[sy, sx] >= thr:
                want[sy, sx] += 1
                if want_first[sy, sx] < 0:
                    want_first[sy, sx] = k
        assert np.array_equal(count, want)
        assert np.array_equal(vmax, want_vmax)
        assert np.array_equal(first, want_first)


def test_first_is_the_smallest_index_in_view(oracle):
    rng = np.random.default_rng(74)
    for occ, srcs, R, thr, sh in cases():
        fields = fields_of(oracle, occ, srcs)
        views = random_views(rng, len(srcs), R)
        _, first, count = fold_view(fields, srcs, views, thr, R, sh)
        ny, nx = occ.shape
        hits = np.stack([m & (f >= thr) & writes_mask(nx, ny, int(sx), int(sy)) for f, (sx, sy), m in
                         zip(fields, srcs, view_masks(occ.shape, srcs, views, R, sh))])
        assert np.array_equal(count, hits.sum(0).astype(np.uint32))
        assert np.array_equal(first, np.where(hits.any(0), hits.argmax(0), -1).astype(np.int32))


def test_new_symbols_are_exported():
    import visibility_heuristic_path_planner_b200 as vhp
    lib = vhp.load_library()
    for name in ("vhp_visibility_merge_view_batch", "vhp_visibility_merge_view_batch_dev"):
        assert hasattr(lib, name)
    assert hasattr(vhp.Context, "visibility_merge_view_batch")
    assert hasattr(vhp.Context, "visibility_merge_view_batch_dev")
