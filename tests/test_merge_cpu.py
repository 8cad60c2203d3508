"""The definition of the merged visibility of a set of light sources (vhp_visibility_merge_batch), pinned on
the CPU oracle against the planner goldens: the element-wise max of computeVisibility over the planner's
light sources lightSources_[0..nb) is visibility_global_, and "the first of those sources whose sweep WRITES
the cell with a value >= threshold" is cameFrom_, bit for bit."""
import hashlib

import numpy as np

from conftest import load_golden

NO_PARENT_U64 = 10**15


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def writes_mask(nx, ny, sx, sy):
    """Cells a sweep from (sx, sy) writes: all but column 0 (unless sx == 0) and row 0 (unless sy == 0)."""
    w = np.ones((ny, nx), bool)
    if sx != 0:
        w[:, 0] = False
    if sy != 0:
        w[0, :] = False
    return w


def fold_fields(fields, srcs, thr, shape, writes_rule=True):
    """vmax / first / count of one group from its fp64 fields (K, ny, nx), sources in group order."""
    ny, nx = shape
    vmax = np.zeros((ny, nx))
    first = np.full((ny, nx), -1, np.int32)
    count = np.zeros((ny, nx), np.uint32)
    for k, (f, (sx, sy)) in enumerate(zip(fields, srcs)):
        vmax = np.maximum(vmax, f)
        hit = f >= thr
        if writes_rule:
            hit &= writes_mask(nx, ny, int(sx), int(sy))
        first[(first < 0) & hit] = k
        count += hit
    return vmax, first, count


def oracle_fold(oracle, occ, srcs, thr, writes_rule=True):
    occ = np.asarray(occ, np.float64)
    fields = [oracle.compute_visibility(occ, int(sx), int(sy)) for sx, sy in srcs]
    return fold_fields(fields, srcs, thr, occ.shape, writes_rule)


def came_u64(first):
    out = first.astype(np.int64)
    out[out < 0] = NO_PARENT_U64
    return out.astype(np.uint64)


def planner_cases(oracle):
    """(name, occ, light sources [0..nb), threshold, vg, came) of every planner golden that sweeps."""
    g = load_golden("planner.npz")
    for seed in range(1, 7):
        st, nb = g[f"s101_{seed}_status"]
        if nb > 0:
            occ = oracle.generate_environment(101, 101, 10, 10, 20, 10, 20, seed)
            yield (f"s101_{seed}", occ, g[f"s101_{seed}_ls"][:nb], 0.25, g[f"s101_{seed}_vg"], g[f"s101_{seed}_came"])
    for k in range(len(g["extra_cases"])):
        st, nb = g[f"extra_{k}_status"]
        if nb > 0:
            yield (f"extra_{k}", g[f"extra_{k}_occ"], g[f"extra_{k}_ls"][:nb], float(g["extra_thr"][k]),
                   g[f"extra_{k}_vg"], g[f"extra_{k}_came"])


def test_fold_reproduces_planner_goldens(oracle):
    names = []
    for name, occ, ls, thr, vg, came in planner_cases(oracle):
        vmax, first, count = oracle_fold(oracle, occ, ls, thr)
        assert np.array_equal(vmax, vg), name
        assert np.array_equal(came_u64(first), came), name
        assert ((count > 0) == (first >= 0)).all() and count.max() <= len(ls)
        names.append(name)
    # every case that sweeps, including thr = 0.0 (extra_3) and the stall to max_iter (extra_4)
    assert names == [f"s101_{s}" for s in range(2, 7)] + [f"extra_{k}" for k in range(5)]


def test_fold_reproduces_maze5_shas(oracle):
    g = load_golden("maze5.npz")
    ny, nx = g["shape"]
    occ = np.unpackbits(g["occ_bits"])[: ny * nx].reshape(ny, nx)
    for tag, thr, want_nb in (("thr020", 0.2, 112), ("thr025", 0.25, 251)):
        st, nb = g[f"{tag}_status"]
        assert nb == want_nb
        vmax, first, _ = oracle_fold(oracle, occ, g[f"{tag}_ls"][:nb], thr)
        assert [sha(vmax), sha(came_u64(first))] == list(g[f"{tag}_sha"][:2]), tag


def test_writes_rule_matters_at_threshold_zero(oracle):
    """With thr = 0.0 every cell passes `v >= thr`; the reference never visits column 0 / row 0 of a sweep
    from elsewhere, so without the "writes" rule the first source wrongly claims them."""
    g = load_golden("planner.npz")
    k = 3
    assert float(g["extra_thr"][k]) == 0.0
    st, nb = g[f"extra_{k}_status"]
    occ, ls = g[f"extra_{k}_occ"], g[f"extra_{k}_ls"][:nb]
    _, naive, _ = oracle_fold(oracle, occ, ls, 0.0, writes_rule=False)
    _, first, _ = oracle_fold(oracle, occ, ls, 0.0)
    assert not np.array_equal(came_u64(naive), g[f"extra_{k}_came"])
    assert np.array_equal(came_u64(first), g[f"extra_{k}_came"])
