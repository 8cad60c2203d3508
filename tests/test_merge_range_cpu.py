"""The definition of range-limited merged visibility (vhp_visibility_merge_range_batch), pinned on the CPU oracle:
the merge of vhp_visibility_merge_batch where source k only contributes to the cells of its range, the box
|dx|, |dy| <= R (the cells of its vhp_visibility_window_batch window) or the disk dx^2 + dy^2 <= R^2.  vmax is the
max of the fields masked to each range, and first / count take the merge's "writes" rule narrowed to the range."""
import numpy as np

from conftest import load_golden
from test_merge_cpu import came_u64, planner_cases, sha, writes_mask
from test_window_cpu import box_mask, seeded_cases, window_of

THRS = (0.5, 1e-9, 0.0, -1.0)


def range_mask(nx, ny, sx, sy, R, disk):
    """Cells in the range of a source at (sx, sy): the box, and for the disk dx^2 + dy^2 <= R^2 as well."""
    m = box_mask(nx, ny, sx, sy, R)
    if disk:
        ys, xs = np.mgrid[0:ny, 0:nx]
        m &= (xs - sx) ** 2 + (ys - sy) ** 2 <= R * R
    return m


def fold_range(fields, srcs, thr, shape, R, disk):
    """vmax / first / count of one group from its full fp64 fields (K, ny, nx), sources in group order."""
    ny, nx = shape
    vmax = np.zeros((ny, nx))
    first = np.full((ny, nx), -1, np.int32)
    count = np.zeros((ny, nx), np.uint32)
    for k, (f, (sx, sy)) in enumerate(zip(fields, srcs)):
        m = range_mask(nx, ny, int(sx), int(sy), R, disk)
        vmax = np.maximum(vmax, np.where(m, f, 0.0))
        hit = m & (f >= thr) & writes_mask(nx, ny, int(sx), int(sy))
        first[(first < 0) & hit] = k
        count += hit
    return vmax, first, count


def fold_windows(windows, srcs, thr, shape, R):
    """The same for the box, from (2R+1)^2 windows alone: each window placed back on the grid and folded."""
    ny, nx = shape
    W = 2 * R + 1
    vmax = np.zeros((ny, nx))
    first = np.full((ny, nx), -1, np.int32)
    count = np.zeros((ny, nx), np.uint32)
    for k, (w, (sx, sy)) in enumerate(zip(windows, srcs)):
        x0, y0 = int(sx) - R, int(sy) - R
        xa, xb, ya, yb = max(x0, 0), min(x0 + W, nx), max(y0, 0), min(y0 + W, ny)
        sub = w[ya - y0:yb - y0, xa - x0:xb - x0]
        wr = writes_mask(nx, ny, int(sx), int(sy))[ya:yb, xa:xb]
        vmax[ya:yb, xa:xb] = np.maximum(vmax[ya:yb, xa:xb], sub)
        hit = (sub >= thr) & wr
        f = first[ya:yb, xa:xb]
        f[(f < 0) & hit] = k
        count[ya:yb, xa:xb] += hit.astype(np.uint32)
    return vmax, first, count


def seeded_groups():
    """(occ, sources, R): the maps and radii of the window tests; the case's source, four random ones and a
    duplicate of the first."""
    rng = np.random.default_rng(505)
    for occ, sx, sy, R in seeded_cases():
        ny, nx = occ.shape
        srcs = [(sx, sy)] + [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(4)] + [(sx, sy)]
        yield occ, np.array(srcs, np.int32), R


def fields_of(oracle, occ, srcs):
    return [oracle.compute_visibility(occ, int(sx), int(sy)) for sx, sy in srcs]


def test_box_beyond_the_map_is_the_merge_planner_goldens(oracle):
    n = 0
    for name, occ, ls, thr, vg, came in planner_cases(oracle):
        occ = np.asarray(occ, np.float64)
        ny, nx = occ.shape
        vmax, first, _ = fold_range(fields_of(oracle, occ, ls), ls, thr, occ.shape, max(nx, ny) - 1, False)
        assert np.array_equal(vmax, vg), name
        assert np.array_equal(came_u64(first), came), name
        n += 1
    assert n == 10


def test_box_beyond_the_map_is_the_merge_maze5_shas(oracle):
    g = load_golden("maze5.npz")
    ny, nx = g["shape"]
    occ = np.unpackbits(g["occ_bits"])[: ny * nx].reshape(ny, nx).astype(np.float64)
    for tag, thr in (("thr020", 0.2), ("thr025", 0.25)):
        st, nb = g[f"{tag}_status"]
        ls = g[f"{tag}_ls"][:nb]
        vmax, first, _ = fold_range(fields_of(oracle, occ, ls), ls, thr, occ.shape, int(max(nx, ny)) - 1, False)
        assert [sha(vmax), sha(came_u64(first))] == list(g[f"{tag}_sha"][:2]), tag


def test_box_is_the_fold_of_the_cropped_windows(oracle):
    for occ, srcs, R in seeded_groups():
        fields = fields_of(oracle, occ, srcs)
        windows = [window_of(f, int(sx), int(sy), R) for f, (sx, sy) in zip(fields, srcs)]
        for thr in THRS:
            want = fold_windows(windows, srcs, thr, occ.shape, R)
            got = fold_range(fields, srcs, thr, occ.shape, R, False)
            for a, b in zip(got, want):
                assert np.array_equal(a, b), (occ.shape, R, thr)


def test_radius_zero_covers_the_source_cells_only(oracle):
    for occ, srcs, _ in seeded_groups():
        ny, nx = occ.shape
        free = [occ[sy, sx] != 0 for sx, sy in srcs]
        on = np.zeros((ny, nx), np.uint32)
        for (sx, sy), fr in zip(srcs, free):
            on[sy, sx] += fr
        for disk in (False, True):
            vmax, first, count = fold_range(fields_of(oracle, occ, srcs), srcs, 0.5, occ.shape, 0, disk)
            assert np.array_equal(count, on)
            assert np.array_equal(vmax, (on > 0).astype(np.float64))
            want_first = np.full((ny, nx), -1, np.int32)
            for k in range(len(srcs) - 1, -1, -1):
                if free[k]:
                    want_first[srcs[k][1], srcs[k][0]] = k
            assert np.array_equal(first, want_first)


def test_outputs_depend_on_nothing_outside_the_boxes(oracle):
    rng = np.random.default_rng(17)
    for occ, srcs, R in seeded_groups():
        ny, nx = occ.shape
        union = np.zeros((ny, nx), bool)
        for sx, sy in srcs:
            union |= box_mask(nx, ny, int(sx), int(sy), R)
        other = np.where(union, occ, rng.integers(0, 2, occ.shape).astype(np.float64))
        fa, fb = fields_of(oracle, occ, srcs), fields_of(oracle, other, srcs)
        for disk in (False, True):
            for thr in (0.5, 0.0):
                a = fold_range(fa, srcs, thr, occ.shape, R, disk)
                b = fold_range(fb, srcs, thr, occ.shape, R, disk)
                for x, y in zip(a, b):
                    assert np.array_equal(x, y), (occ.shape, R, disk, thr)


def test_disk_differs_from_box(oracle):
    """The disk's mask matters: on this seeded family the coverage counts of disk and box differ in 30 of the 60
    cases (in the others no cell of a box outside its disk reaches the threshold, or none lies on the grid)."""
    differ = 0
    for occ, srcs, R in seeded_groups():
        fields = fields_of(oracle, occ, srcs)
        box = fold_range(fields, srcs, 0.5, occ.shape, R, False)
        disk = fold_range(fields, srcs, 0.5, occ.shape, R, True)
        assert (disk[2] <= box[2]).all() and (disk[0] <= box[0]).all()
        differ += not np.array_equal(disk[2], box[2])
    assert differ == 30
