"""The planner's next-source choice when several cells tie on h, against the reference's loop order.

heap_->top() is the first pushed cell with the minimum h: the push order is Q1..Q4, i outer, j inner, and a cell on
an axis counts in the first quadrant that visits it.  The kernels stand for it with a key quadrant << 40 | i << 20 | j
(planner_common.cuh) and reduce (h bits, key) lexicographically in five places (the persistent CTA, the batch-wide
first sweep, the grid route's strip epilogue, the strip-partitioned planner, every warp instance).  The key only
decides something when two cells have bit-identical h, which random maps almost never give.  This file builds maps
where they do -- mirrored about the source's column, its row, both, or the main diagonal, and dark cells on the
segment between start and end at threshold 0 -- and checks, without a GPU:

  - the key, restated from the kernel, sorts the cells of every source on every small grid into the order the
    reference's four loop nests first visit them;
  - for every case the GPU tests run (test_gpu_planner_ties.py), a witness from the oracle stepped one sweep at a
    time: at each iteration the cells at the minimum of the recomputed h, their quadrants, and whether the first
    pushed one is not the one with the smallest linear index; the oracle's pick is the first pushed of them;
  - the cases together tie across every pair of quadrants, within one quadrant at (i, j) against (j, i), an axis
    cell against an off-axis one, at the first sweep and at later ones, in one row and across rows, and at least
    once with a winner that is not the smallest index."""
import itertools

import numpy as np
import pytest

from conftest import rect_map
from visibility_heuristic_path_planner_b200.sharding import shard_bounds

NO_PARENT = 10**15
SYM_THR, SYM_ITER = 0.3, 25  # symmetric maps: the threshold and iteration cap of every case
LINE_THR, LINE_ITER = 0.0, 12  # start and end on one row or column


# ---- maps mirrored about the source ------------------------------------------------------------------------------

def mirror_about_column(left):
    """left: (ny, a + 1); its last column is the axis, the result is (ny, 2a + 1)"""
    occ = np.concatenate([left, left[:, -2::-1]], axis=1)
    assert np.array_equal(occ, occ[:, ::-1])
    return occ


def mirror_about_row(low):
    """low: (a + 1, nx); its last row is the axis, the result is (2a + 1, nx)"""
    occ = mirror_about_column(low.T).T.copy()
    assert np.array_equal(occ, occ[::-1, :])
    return occ


def mirror_about_both(quarter):
    occ = mirror_about_row(mirror_about_column(quarter))
    assert np.array_equal(occ, occ[::-1, :]) and np.array_equal(occ, occ[:, ::-1])
    return occ


def transpose_symmetric(occ):
    """The lower triangle (the diagonal included) of a square map reflected onto the upper one"""
    sym = np.tril(occ) + np.tril(occ, -1).T
    assert np.array_equal(sym, sym.T)
    return sym


def mirror_rows_about(occ, r):
    """Rows r - d := rows r + d wherever both exist: symmetric about row r in the band it allows (the rest of the
    map unchanged); for the strip-partitioned planner, whose strip boundaries are not at the map's middle row"""
    occ = occ.copy()
    d = min(r, occ.shape[0] - 1 - r)
    occ[r - d:r] = occ[r + d:r:-1]
    assert np.array_equal(occ[r - d:r + d + 1], occ[r - d:r + d + 1][::-1])
    return occ


def free(occ, *cells):
    occ = occ.copy()
    for x, y in cells:
        occ[y, x] = 1
    return occ


# ---- the push order ----------------------------------------------------------------------------------------------

def push_key(x, y, sx, sy):
    """planner_common.cuh's (quadrant, i, j) rule, restated"""
    dx, dy = x - sx, y - sy
    if dx >= 0 and dy >= 0:
        q, i, j = 0, dx, dy
    elif dx < 0 and dy >= 0:
        q, i, j = 1, -dx, dy
    elif dx <= 0 and (dx < 0 or sx >= 1):
        q, i, j = 2, -dx, -dy
    else:
        q, i, j = 3, dx, -dy
    return q << 40 | i << 20 | j


def quadrant(key):
    return key >> 40


def first_visits(nx, ny, sx, sy):
    """The reference's loop nests spelled out: Q1..Q4, i outer, j inner; Q2 / Q3 stop at X = 1, Q3 / Q4 at Y = 1.
    Returns [(x, y, quadrant)] in the order cells are first visited."""
    nests = ((1, 1, nx - sx, ny - sy), (-1, 1, sx, ny - sy), (-1, -1, sx, sy), (1, -1, nx - sx, sy))
    out, seen = [], set()
    for q, (dirx, diry, ni, nj) in enumerate(nests):
        for i in range(ni):
            for j in range(nj):
                c = (sx + dirx * i, sy + diry * j)
                if c not in seen:
                    seen.add(c)
                    out.append(c + (q,))
    return out


def visited_mask(nx, ny, sx, sy):
    """Cells a sweep from (sx, sy) visits: all but column 0 when sx > 0 and row 0 when sy > 0"""
    m = np.ones((ny, nx), bool)
    if sx > 0:
        m[:, 0] = False
    if sy > 0:
        m[0, :] = False
    return m


@pytest.mark.parametrize("nx, ny", list(itertools.product(range(1, 10), range(1, 8))))
def test_key_order_is_first_visit_order(nx, ny):
    for sx in range(nx):
        for sy in range(ny):
            order = first_visits(nx, ny, sx, sy)
            cells = [(x, y) for x, y, _ in order]
            assert sorted(cells, key=lambda c: push_key(c[0], c[1], sx, sy)) == cells, (nx, ny, sx, sy)
            assert [quadrant(push_key(x, y, sx, sy)) for x, y, _ in order] == [q for _, _, q in order]
            m = visited_mask(nx, ny, sx, sy)
            assert sorted(cells) == sorted((int(x), int(y)) for y, x in np.argwhere(m)), (nx, ny, sx, sy)


# ---- the oracle stepped one sweep at a time ----------------------------------------------------------------------

def eval_d(xs, ys, x, y):
    """include/solver/visibilityBasedSolver.h:112-115 on integer coordinates (every operand exact)"""
    return np.sqrt((xs - x).astype(np.float64) ** 2 + ((ys - y) ** 2).astype(np.float64))


def stepped(oracle, occ, start, end, thr, max_iter):
    """solve() as a loop of update_visibility calls.  Per sweep: the recomputed heuristic over the cells it pushes,
    the cells at its minimum and the oracle's pick.  Returns (light sources, [per-iteration record])."""
    occ = np.asarray(occ, np.float64)
    ny, nx = occ.shape
    ys, xs = np.mgrid[0:ny, 0:nx]
    scale = np.sqrt(float(ny * ny + nx * nx))
    vg, came = np.zeros((ny, nx)), np.full((ny, nx), NO_PARENT, np.uint64)
    came[start[1], start[0]] = 0
    ls, src, recs = [tuple(start)], tuple(start), []
    d_end = eval_d(xs, ys, *end)
    while vg[end[1], end[0]] <= thr:
        nb = len(ls) - 1
        _, top, top_h, _ = oracle.update_visibility(occ, src, end, thr, vg, came, np.array(ls), nb)
        pushed = visited_mask(nx, ny, *src) & (vg >= thr)
        par = np.array(ls)[came[pushed].astype(np.int64)]
        h = np.full((ny, nx), np.inf)
        h[pushed] = scale * vg[pushed] + (d_end[pushed] + eval_d(xs[pushed], ys[pushed], par[:, 0], par[:, 1]))
        hmin = h.min()
        tied = [(int(x), int(y)) for y, x in np.argwhere(h == hmin)]  # row-major: linear index order
        keys = [push_key(x, y, *src) for x, y in tied]
        first = tied[int(np.argmin(keys))]
        assert top_h == hmin and top == first, (nb, src, top, top_h, first, hmin)
        recs.append(dict(nb=nb, src=src, tied=tied, keys=keys, winner=first))
        src = top
        ls.append(top)
        if len(ls) - 1 > max_iter:
            break
    return ls, recs


def tie_classes(rec):
    """The kinds of tie one iteration's record shows (nothing if a single cell holds the minimum)"""
    tied, keys, (sx, sy) = rec["tied"], rec["keys"], rec["src"]
    if len(tied) < 2:
        return set()
    out = {"nb=0" if rec["nb"] == 0 else "nb>=1"}
    quads = sorted({quadrant(k) for k in keys})
    out |= {f"Q{a + 1}/Q{b + 1}" for a, b in itertools.combinations(quads, 2)}
    ij = {(quadrant(k), (k >> 20) & 0xFFFFF, k & 0xFFFFF) for k in keys}
    if any(i != j and (q, j, i) in ij for q, i, j in ij):
        out.add("(i,j)/(j,i)")
    on_axis = [x == sx or y == sy for x, y in tied]
    if any(on_axis) and not all(on_axis):
        out.add("axis/off-axis")
    rows = [y for _, y in tied]
    if len(set(rows)) > 1:
        out.add("rows differ")
    if len(set(rows)) < len(rows):
        out.add("same row")
    if rec["winner"] != tied[0]:
        out.add("winner not smallest index")
    return out


ALL_CLASSES = {"Q1/Q2", "Q1/Q4", "Q2/Q3", "Q3/Q4", "Q1/Q3", "Q2/Q4", "(i,j)/(j,i)", "axis/off-axis", "nb=0",
               "nb>=1", "rows differ", "same row", "winner not smallest index"}


# ---- the cases ---------------------------------------------------------------------------------------------------

N = 61  # every symmetric case is 61 x 61, so each group runs as one batch
A = N // 2


def symmetric_map(family, seed):
    """A 61 x 61 map of one family: random rectangles on the part that is mirrored"""
    if family == "column":
        return mirror_about_column(rect_map(A + 1, N, 30, seed, 2, 7))
    if family == "row":
        return mirror_about_row(rect_map(N, A + 1, 30, seed, 2, 7))
    if family == "both":
        return mirror_about_both(rect_map(A + 1, A + 1, 30, seed, 2, 7))
    return transpose_symmetric(rect_map(N, N, 60, seed, 2, 7))


# (family, seed, start, end): the end on the symmetry axis above (larger y), below, left and right of the start, and
# sources on each border: sx = 0 (Q2 and Q3 empty), sy = 0, the last column and the last row.  Every seed is one
# whose witness ties (test_every_case_ties).
SYMMETRIC = [
    ("column", 103, (A, 8), (A, 52)), ("column", 103, (A, 52), (A, 8)), ("column", 101, (A, 30), (A, 55)),
    ("row", 100, (8, A), (52, A)), ("row", 102, (52, A), (8, A)), ("row", 101, (30, A), (3, A)),
    ("both", 100, (A, A), (A, 56)), ("both", 100, (A, A), (A, 4)), ("both", 100, (A, A), (4, A)),
    ("both", 100, (A, A), (56, A)),
    ("transpose", 108, (6, 6), (54, 54)), ("transpose", 100, (50, 50), (9, 9)), ("transpose", 100, (30, 30), (58, 58)),
    ("row", 102, (0, A), (57, A)), ("column", 103, (A, 0), (A, 57)), ("row", 104, (N - 1, A), (3, A)),
    ("column", 117, (A, N - 1), (A, 3)),
]


def symmetric_cases():
    """(name, occ, start, end) of SYMMETRIC"""
    return [(f"{family}{seed}_{start[0]}_{start[1]}_{end[0]}_{end[1]}", free(symmetric_map(family, seed), start, end),
             start, end) for family, seed, start, end in SYMMETRIC]


def blocked_segment(occ, start, end, step):
    """An obstacle every `step` cells of the row or column segment between start and end (the end in the dark)"""
    occ = occ.copy()
    (sx, sy), (ex, ey) = start, end
    for t in range(3, max(abs(ex - sx), abs(ey - sy)), step):
        occ[sy + t * np.sign(ey - sy), sx + t * np.sign(ex - sx)] = 0
    return occ


def line_cases():
    """(name, occ, start, end) at threshold 0: start and end on one row or column of a map with no symmetry.  A dark
    cell on the segment has vg = 0 and d_end + d_parent = |SE|, an integer, so all of them tie."""
    cases = []
    for seed, (start, end) in zip((61, 62, 63, 64), (((5, 20), (55, 20)), ((55, 40), (5, 40)), ((17, 4), (17, 57)),
                                                     ((44, 57), (44, 4)))):
        cases.append((f"line{seed}", free(blocked_segment(rect_map(N, N, 30, seed, 2, 7), start, end, 6), start, end),
                      start, end))
    return cases


def big_line_cases():
    """The same on a 1000 x 1000 map and on a 12000 x 48 one (too wide for one CTA: the grid route by default)"""
    big = ((900, 500), (40, 500))
    wide = ((11900, 21), (30, 21))
    return [("line1000", free(blocked_segment(rect_map(1000, 1000, 400, 1000, 4, 40), *big, 97), *big)) + big,
            ("line12000x48", free(blocked_segment(rect_map(12000, 48, 300, 12000, 4, 30), *wide, 1009), *wide)) + wide]


GIANT_NX, GIANT_NY = 150, 170  # five strips of 34 rows at most (a strip holds at least one 32-row tile row)
GIANT_STRIPS = (1, 2, 3, 5)
# (strips, seed, ends): the map mirrored about the first row of strip 1 (the middle row for one strip); start and end
# on that row, the end to the right or to the left
GIANT = [(1, 1, "right"), (1, 1, "left"), (2, 1, "right"), (2, 1, "left"), (3, 1, "right"), (3, 1, "left"),
         (5, 1, "right"), (5, 2, "left")]


def giant_case(nstrips, seed, ends):
    """(occ, start, end, strip row ranges): a tie between rows r - d and r + d is a tie between two strips"""
    bounds = [shard_bounds(GIANT_NY, k, nstrips) for k in range(nstrips)]
    r = bounds[1][0] if nstrips > 1 else GIANT_NY // 2
    start, end = ((12, r), (137, r)) if ends == "right" else ((137, r), (12, r))
    occ = free(mirror_rows_about(rect_map(GIANT_NX, GIANT_NY, 120, seed, 2, 9), r), start, end)
    return occ, start, end, bounds


def strip_of(y, bounds):
    return next(k for k, (lo, hi) in enumerate(bounds) if lo <= y < hi)


def giant_cases():
    """(name, occ, start, end, strip row ranges) of GIANT"""
    return [(f"giant{n}_{seed}_{ends}",) + giant_case(n, seed, ends) for n, seed, ends in GIANT]


@pytest.fixture(scope="module")
def witnesses(oracle):
    """name -> the stepped oracle's per-iteration records, for every case the GPU tests run"""
    out = {}
    giant = [c[:4] for c in giant_cases()]
    for cases, thr, mi in ((symmetric_cases(), SYM_THR, SYM_ITER), (line_cases(), LINE_THR, LINE_ITER),
                           (big_line_cases(), LINE_THR, LINE_ITER), (giant, SYM_THR, SYM_ITER)):
        for name, occ, start, end in cases:
            ls, recs = stepped(oracle, occ, start, end, thr, mi)
            ref = oracle.solve(occ, start, end, thr, mi)
            nb = ref["nb_of_sources"]
            n = nb + 1 if ref["status"] == 5 else nb  # (at status 0 the last entry is the end)
            assert len(ls) == nb + 1 and np.array_equal(np.array(ls[:n]), ref["light_sources"][:n]), name
            out[name] = recs
    return out


def test_symmetric_builders():
    rng = np.random.default_rng(0)
    for ny, nx in ((1, 1), (3, 5), (8, 2)):
        m = rng.integers(0, 2, (ny, nx)).astype(np.float64)
        mirror_about_column(m), mirror_about_row(m), mirror_about_both(m)
        assert mirror_about_both(m).shape == (2 * ny - 1, 2 * nx - 1)
        transpose_symmetric(rng.integers(0, 2, (nx, nx)).astype(np.float64))
        mirror_rows_about(rng.integers(0, 2, (7, nx)).astype(np.float64), ny % 7)


def test_transpose_symmetric_field(oracle):
    """On a transpose-symmetric map, from a source on the diagonal, the field equals its transpose over Q1 and Q3:
    transposing maps each of them onto itself with i and j swapped, the i > j branch onto the j > i one, and the
    diagonal rule (vis(k, k) = the stale value of (k, k - 1)) onto itself by induction.  Q2 and Q4 map onto each
    other, and there the diagonal rule does not: Q2's diagonal copies its (i, i - 1), whose mirror is Q4's
    (i - 1, i), while Q4's diagonal copies Q4's (i, i - 1).  So a tie across Q2 / Q4 on such a map is not
    guaranteed; one seed shows the difference."""
    asymmetric = 0
    for seed in (100, 101, 108):
        occ = symmetric_map("transpose", seed)
        for s in (0, 6, A, N - 1):
            vis = oracle.compute_visibility(free(occ, (s, s)), s, s)
            ys, xs = np.mgrid[0:N, 0:N]
            q13 = (xs - s) * (ys - s) >= 0
            assert np.array_equal(vis[q13], vis.T[q13]), (seed, s)
            asymmetric += not np.array_equal(vis, vis.T)
    assert asymmetric == 1  # seed 101 from (30, 30)


def test_every_case_ties(witnesses):
    """Every case, pinned by its seed, has two or more cells at the minimum h at one iteration or more"""
    ties = {name: [r["nb"] for r in recs if len(r["tied"]) > 1] for name, recs in witnesses.items()}
    assert all(ties.values()), {k: v for k, v in ties.items() if not v}


def test_cases_cover_every_tie_class(witnesses):
    seen = set()
    for recs in witnesses.values():
        for r in recs:
            seen |= tie_classes(r)
    assert seen >= ALL_CLASSES, ALL_CLASSES - seen


def test_giant_ties_cross_strip_boundaries(witnesses):
    """Where the map has two or more strips, cells of two strips tie: the cross-strip minimum decides"""
    for name, occ, start, end, bounds in giant_cases():
        if len(bounds) > 1:
            assert any(len({strip_of(y, bounds) for _, y in r["tied"]}) > 1 for r in witnesses[name]), name
