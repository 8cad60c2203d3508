"""The definition of range-limited visibility (vhp_visibility_window_batch), pinned on the CPU oracle: the
(2R+1)^2 window centred on the source is the crop of computeVisibility's full field, 0 outside the grid.
In each quadrant cell (i, j) depends only on cells with offsets <= (i, j) component-wise, so the Chebyshev box
|dx| <= R, |dy| <= R around the source is closed under "upstream": the window depends on nothing outside it.
It is NOT the sweep of the map cropped to the box: the never-written border (column 0 / row 0 of the grid)
sits at absolute coordinates, and a cropped map moves it to the box's edge."""
import numpy as np


def window_of(field, sx, sy, R):
    """(2R+1, 2R+1) window of a (ny, nx) field centred on (sx, sy); cells outside the grid are 0."""
    ny, nx = field.shape
    w = 2 * R + 1
    out = np.zeros((w, w), field.dtype)
    x0, y0 = sx - R, sy - R
    xa, xb = max(x0, 0), min(x0 + w, nx)
    ya, yb = max(y0, 0), min(y0 + w, ny)
    out[ya - y0:yb - y0, xa - x0:xb - x0] = field[ya:yb, xa:xb]
    return out


def box_mask(nx, ny, sx, sy, R):
    m = np.zeros((ny, nx), bool)
    m[max(sy - R, 0):sy + R + 1, max(sx - R, 0):sx + R + 1] = True
    return m


def seeded_cases(n=60):
    """(occ, sx, sy, R): random rectangle maps of 1..70 cells per side; sources on corners and edges first, then
    anywhere; R = 0, R beyond the larger side, and R in [0, 40) otherwise."""
    rng = np.random.default_rng(2024)
    for k in range(n):
        nx, ny = int(rng.integers(1, 71)), int(rng.integers(1, 71))
        occ = np.ones((ny, nx))
        for _ in range(int(rng.integers(0, nx * ny // 60 + 2))):
            x, y = int(rng.integers(0, nx)), int(rng.integers(0, ny))
            occ[y:y + int(rng.integers(1, 8)), x:x + int(rng.integers(1, 8))] = 0
        corners = [(0, 0), (nx - 1, 0), (0, ny - 1), (nx - 1, ny - 1), (nx // 2, 0), (0, ny // 2)]
        sx, sy = corners[k] if k < len(corners) else (int(rng.integers(0, nx)), int(rng.integers(0, ny)))
        R = 0 if k % 10 == 7 else (max(nx, ny) + int(rng.integers(0, 5)) if k % 10 == 8 else int(rng.integers(0, 40)))
        yield occ, sx, sy, R


def test_window_of_pads_with_zeros():
    f = np.arange(12, dtype=np.float64).reshape(3, 4) + 1
    w = window_of(f, 0, 2, 2)
    assert w.shape == (5, 5)
    assert np.array_equal(w[:3, 2:], f[:, :3]) and not w[3:].any() and not w[:, :2].any()
    assert np.array_equal(window_of(f, 1, 1, 0), [[f[1, 1]]])


def test_window_depends_on_nothing_outside_it(oracle):
    rng = np.random.default_rng(7)
    n = 0
    for occ, sx, sy, R in seeded_cases():
        ny, nx = occ.shape
        want = window_of(oracle.compute_visibility(occ, sx, sy), sx, sy, R)
        inside = box_mask(nx, ny, sx, sy, R)
        for _ in range(2):
            other = np.where(inside, occ, rng.integers(0, 2, occ.shape).astype(np.float64))
            got = window_of(oracle.compute_visibility(other, sx, sy), sx, sy, R)
            assert np.array_equal(got, want), (nx, ny, sx, sy, R)
        n += 1
    assert n == 60


def test_window_is_not_the_sweep_of_the_cropped_map(oracle):
    """Cutting the map to the box and sweeping it from the source's position in the box puts the never-written
    border at the box's edge instead of at column 0 / row 0: on this seeded family that differs from the window
    in 21 of the 38 cases whose box is not the whole map."""
    differ = total = 0
    for occ, sx, sy, R in seeded_cases():
        ny, nx = occ.shape
        x0, y0 = max(sx - R, 0), max(sy - R, 0)
        if x0 == 0 and y0 == 0 and sx + R >= nx - 1 and sy + R >= ny - 1:
            continue  # the box is the whole map
        want = window_of(oracle.compute_visibility(occ, sx, sy), sx, sy, R)
        sub = np.ascontiguousarray(occ[y0:sy + R + 1, x0:sx + R + 1])
        crop = oracle.compute_visibility(sub, sx - x0, sy - y0)
        full = np.zeros_like(want)
        full[y0 - (sy - R):y0 - (sy - R) + sub.shape[0], x0 - (sx - R):x0 - (sx - R) + sub.shape[1]] = crop
        total += 1
        differ += not np.array_equal(full, want)
    assert (differ, total) == (21, 38)
