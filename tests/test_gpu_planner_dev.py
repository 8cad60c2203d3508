"""The device entry point of the planner (vhp_planner_batch_dev) against the oracle and the goldens,
and the parts of the planner the host-form tests of test_gpu_planner.py do not reach: optional
outputs, ls_cap above max_iter + 2, the chunk edges of the host staging (2 GiB) and of the device
workspace (32 GiB), prepared maps, and the loop modes and captured graph of the grid route.

Where the oracle can run every check is exact: fp64 outputs bit for bit, fp32 fields equal to the
fp64 value rounded once.  Outputs the call is expected to write start as a sentinel (-7 / NaN), so an
output left unwritten fails."""
import hashlib
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import load_golden, rect_map

pytestmark = pytest.mark.gpu
NO_PARENT_U64 = 10**15
SMALL = ("status", "nb_sources", "light_sources", "path_len", "path_n", "path")
FIELDS = ("vg", "came", "vis")
ALL = SMALL + FIELDS


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def came_u64(came_i32):
    out = came_i32.astype(np.int64)
    out[out < 0] = NO_PARENT_U64
    return out.astype(np.uint64)


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def make_ctx(vhp, torch, route="default"):
    """A context on a stream of its own; `c.stream` is where the tests enqueue their torch work.
    Routes as in test_gpu_planner.py: cta (one persistent CTA per problem), first (the first sweep of
    every problem batch-wide, forced with VHP_PLANNER_FIRST=2 / VHP_PLANNER_ROUNDS=3, read at context
    creation), grid (one problem at a time on the whole GPU, set_grid_sweep(2)); default = library
    defaults."""
    if route == "first":
        os.environ["VHP_PLANNER_FIRST"] = "2"
        os.environ["VHP_PLANNER_ROUNDS"] = "3"
    stream = torch.cuda.Stream(torch.device("cuda", 0))
    try:
        c = vhp.torch_context(0, stream)
    finally:
        os.environ.pop("VHP_PLANNER_FIRST", None)
        os.environ.pop("VHP_PLANNER_ROUNDS", None)
    if route != "default":
        c.set_grid_sweep(2 if route == "grid" else 0)
    c.stream = stream
    return c


@pytest.fixture(scope="module", params=["cta", "first", "grid"])
def ctx(vhp, torch, request):
    c = make_ctx(vhp, torch, request.param)
    yield c
    c.close()


def dev_outputs(torch, n, ny, nx, cap, dtype_f32, which):
    """Sentinel-filled CUDA tensors for the outputs in `which`."""
    d = torch.device("cuda", 0)
    ft = torch.float32 if dtype_f32 else torch.float64
    shapes = dict(status=((n,), torch.int32), nb_sources=((n,), torch.int32),
                  light_sources=((n, cap, 2), torch.int32), path_len=((n,), torch.float64),
                  path_n=((n,), torch.int32), path=((n, cap, 2), torch.int32),
                  vg=((n, ny, nx), ft), came=((n, ny, nx), torch.int32), vis=((n, ny, nx), ft))
    out = {}
    for k in which:
        shp, dt = shapes[k]
        out[k] = torch.full(shp, float("nan") if dt.is_floating_point else -7, dtype=dt, device=d)
    return out


def run_dev(ctx, vhp, torch, occ, se, pmap=None, thr=0.5, max_iter=100, ls_cap=None, dtype=None, which=ALL,
            occ_t=None, out=None):
    """planner_batch_dev on uploaded copies of the inputs; returns the outputs as numpy arrays
    (keys of planner_batch)."""
    dtype = vhp.F64 if dtype is None else dtype
    se = np.ascontiguousarray(se, dtype=np.int32).reshape(-1, 4)
    n = se.shape[0]
    cap = max_iter + 2 if ls_cap is None else ls_cap
    with torch.cuda.stream(ctx.stream):
        if occ_t is None:
            o = np.asarray(occ)
            occ_t = torch.from_numpy(np.ascontiguousarray((o if o.ndim == 3 else o[None]) != 0, np.uint8)).cuda()
        se_t = torch.from_numpy(se).cuda()
        pm_t = None if pmap is None else torch.from_numpy(np.ascontiguousarray(pmap, np.int32)).cuda()
        _, ny, nx = occ_t.shape
        if out is None:
            out = dev_outputs(torch, n, ny, nx, cap, dtype == vhp.F32, which)
        ctx.planner_batch_dev(occ_t, se_t, pm_t, threshold=thr, max_iter=max_iter, ls_cap=ls_cap, dtype=dtype,
                              **out)
        r = {k: v.cpu().numpy() for k, v in out.items()}
    ctx.stream.synchronize()
    return r


def check(r, k, ref, full=True, f32=False):
    """r: result dict, k: problem index, ref: oracle/golden dict (fp64 fields)."""
    st, nb = int(r["status"][k]), int(r["nb_sources"][k])
    assert (st, nb) == (ref["status"], ref["nb_of_sources"]), (k, st, nb, ref["status"], ref["nb_of_sources"])
    if st in (0, 5):
        assert np.array_equal(r["light_sources"][k][: nb + 1], ref["light_sources"]), k
    n = int(r["path_n"][k])
    assert np.array_equal(r["path"][k][:n], ref["path"]), k
    assert r["path_len"][k] == ref["path_length"], k
    if full:
        cast = (lambda a: a.astype(np.float32)) if f32 else (lambda a: a)
        assert np.array_equal(r["vg"][k], cast(ref["vg"])), k
        assert np.array_equal(came_u64(r["came"][k]), ref["came"]), k
        assert np.array_equal(r["vis"][k], cast(ref["vis"])), k


def same_output(a, b, key, k, nb=None, pn=None):
    """Output `key` of problem k equal in two results (light sources up to nb + 1, path up to path_n)."""
    x, y = a[key][k], b[key][k]
    if key == "light_sources":
        x, y = x[: nb + 1], y[: nb + 1]
    elif key == "path":
        x, y = x[:pn], y[:pn]
    assert np.array_equal(x, y), (key, k)


def same_results(a, b, keys, n):
    """(A problem that fails validation (status 1-4) writes no light source.)"""
    for k in range(n):
        nb, pn = int(a["nb_sources"][k]), int(a["path_n"][k])
        for key in keys:
            if key != "light_sources" or int(a["status"][k]) in (0, 5):
                same_output(a, b, key, k, nb, pn)


def maze5():
    g = load_golden("maze5.npz")
    ny, nx = g["shape"]
    occ = np.unpackbits(g["occ_bits"])[: ny * nx].reshape(ny, nx)
    return g, occ, tuple(g["start"]) + tuple(g["end"])


def check_maze(r, k, g, tag):
    st, nb = g[f"{tag}_status"]
    assert (int(r["status"][k]), int(r["nb_sources"][k])) == (st, nb), tag
    assert np.array_equal(r["light_sources"][k][: nb + 1], g[f"{tag}_ls"]), tag
    assert np.array_equal(r["path"][k][: int(r["path_n"][k])], g[f"{tag}_path"]), tag
    assert r["path_len"][k] == g[f"{tag}_len"][0], tag
    if "vg" in r:
        assert [sha(r["vg"][k]), sha(came_u64(r["came"][k])), sha(r["vis"][k])] == list(g[f"{tag}_sha"]), tag


def free_points(occ, n, rng):
    free = np.argwhere(np.asarray(occ) != 0)
    p = free[rng.integers(0, len(free), n)]
    return p[:, 1], p[:, 0]


# ---- the device form against the oracle ---------------------------------------------------------------
def test_dev_goldens_101(ctx, vhp, torch, oracle):
    g = load_golden("planner.npz")
    maps = np.stack([oracle.generate_environment(101, 101, 10, 10, 20, 10, 20, s) for s in range(1, 7)])
    se = np.tile(np.array([5, 5, 95, 95], np.int32), (6, 1))
    for dtype in (vhp.F64, vhp.F32):
        r = run_dev(ctx, vhp, torch, maps, se, pmap=np.arange(6), thr=0.25, max_iter=100, dtype=dtype)
        for k, seed in enumerate(range(1, 7)):
            ref = dict(status=int(g[f"s101_{seed}_status"][0]), nb_of_sources=int(g[f"s101_{seed}_status"][1]),
                       light_sources=g[f"s101_{seed}_ls"], path=g[f"s101_{seed}_path"],
                       path_length=g[f"s101_{seed}_len"][0], vg=g[f"s101_{seed}_vg"],
                       came=g[f"s101_{seed}_came"], vis=g[f"s101_{seed}_vis"])
            check(r, k, ref, f32=dtype == vhp.F32)


def test_dev_extra_cases(ctx, vhp, torch, oracle):
    g = load_golden("planner.npz")
    for k, c in enumerate(g["extra_cases"]):
        occ = g[f"extra_{k}_occ"]
        thr, mi = float(g["extra_thr"][k]), int(c[8])
        ref = oracle.solve(occ.astype(np.float64), (c[4], c[5]), (c[6], c[7]), thr, mi)
        assert ref["status"] == int(g[f"extra_{k}_status"][0]) and ref["path_length"] == g[f"extra_{k}_len"][0]
        for dtype in (vhp.F64, vhp.F32):
            r = run_dev(ctx, vhp, torch, occ, [(c[4], c[5], c[6], c[7])], thr=thr, max_iter=mi, dtype=dtype)
            check(r, 0, ref, f32=dtype == vhp.F32)


def test_dev_maze5(ctx, vhp, torch):
    g, occ, se = maze5()
    for tag, thr in (("thr020", 0.2), ("thr030", 0.3), ("thr025", 0.25)):
        check_maze(run_dev(ctx, vhp, torch, occ, [se], thr=thr, max_iter=250), 0, g, tag)


def test_dev_random_problems(ctx, vhp, torch, oracle):
    """Several maps per call through a device prob_map, both dtypes."""
    rng = np.random.default_rng(4242)
    for trial in range(4):
        nx, ny = int(rng.integers(20, 180)), int(rng.integers(20, 180))
        maps = np.stack([rect_map(nx, ny, int(rng.integers(0, 30)), 900 + 3 * trial + m, 2, 14) for m in range(3)])
        n = 9
        pmap = rng.integers(0, 3, n).astype(np.int32)
        se = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n), rng.integers(0, nx, n),
                       rng.integers(0, ny, n)], axis=1).astype(np.int32)
        thr = float(rng.choice([0.0, 0.2, 0.5, 0.9]))
        refs = [oracle.solve(maps[pmap[k]], se[k][:2], se[k][2:], thr, 10) for k in range(n)]
        for dtype in (vhp.F64, vhp.F32):
            r = run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=thr, max_iter=10, dtype=dtype)
            for k in range(n):
                check(r, k, refs[k], f32=dtype == vhp.F32)


def test_dev_vis_off_16_byte_boundary(ctx, vhp, torch, oracle):
    """An fp64 vis output 8 bytes past a 16-byte boundary at even nx: the planner kernel's scalar
    stores (its paired stores need a 16-byte aligned field)."""
    nx, ny, n = 96, 70, 3
    occ = rect_map(nx, ny, 14, 31, 3, 12)
    rng = np.random.default_rng(5)
    xs, ys = free_points(occ, 2 * n, rng)
    se = np.stack([xs[:n], ys[:n], xs[n:], ys[n:]], axis=1).astype(np.int32)
    with torch.cuda.stream(ctx.stream):
        out = dev_outputs(torch, n, ny, nx, 14, False, ALL)
        buf = torch.full((n * ny * nx + 1,), float("nan"), dtype=torch.float64, device="cuda")
    out["vis"] = buf[1:].view(n, ny, nx)
    assert out["vis"].data_ptr() % 16 == 8
    r = run_dev(ctx, vhp, torch, occ, se, thr=0.3, max_iter=12, out=out)
    for k in range(n):
        check(r, k, oracle.solve(occ, se[k][:2], se[k][2:], 0.3, 12))


# ---- optional outputs ---------------------------------------------------------------------------------
def test_optional_outputs(ctx, vhp, torch, oracle):
    """Each output NULL in turn, only the small ones, only the fields, and no output struct at all:
    what was requested equals the full call's, on every route and in both dtypes."""
    maps = np.stack([oracle.generate_environment(101, 101, 10, 10, 20, 10, 20, s) for s in (2, 3)])
    se = np.array([[5, 5, 95, 95], [5, 5, 95, 95], [50, 10, 12, 90]], np.int32)
    pmap = np.array([0, 1, 1], np.int32)
    for k in range(3):
        for m in range(2):
            maps[m, se[k, 1], se[k, 0]] = maps[m, se[k, 3], se[k, 2]] = 1
    for dtype in (vhp.F64, vhp.F32):
        full = run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=0.25, max_iter=40, dtype=dtype)
        for k in range(3):
            check(full, k, oracle.solve(maps[pmap[k]], se[k][:2], se[k][2:], 0.25, 40), f32=dtype == vhp.F32)
        subsets = [tuple(x for x in ALL if x != skip) for skip in ALL] + [SMALL, FIELDS]
        for which in subsets:
            r = run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=0.25, max_iter=40, dtype=dtype, which=which)
            assert set(r) == set(which)
            same_results(full, r, which, 3)
        # no output struct: the call runs and leaves the context usable
        run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=0.25, max_iter=40, dtype=dtype, which=())
        again = run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=0.25, max_iter=40, dtype=dtype)
        same_results(full, again, ALL, 3)


# ---- ls_cap -------------------------------------------------------------------------------------------
def test_ls_cap_strides(ctx, vhp, torch, oracle):
    """ls_cap = max_iter + 2, + 5 and 3 * (max_iter + 2) in both forms: the light-source and path rows
    of every problem start at q * ls_cap.  Entries past nb + 1 are not compared."""
    nx, ny, mi = 120, 90, 9
    maps = np.stack([rect_map(nx, ny, 25, 71 + m, 3, 15) for m in range(2)])
    rng = np.random.default_rng(12)
    n = 7
    pmap = rng.integers(0, 2, n).astype(np.int32)
    se = np.zeros((n, 4), np.int32)
    for k in range(n):
        xs, ys = free_points(maps[pmap[k]], 2, rng)
        se[k] = (xs[0], ys[0], xs[1], ys[1])
    for thr in (0.9, 0.3):  # (0.9: most problems run into max_iter and fill nb + 1 = max_iter + 2 entries)
        refs = [oracle.solve(maps[pmap[k]], se[k][:2], se[k][2:], thr, mi) for k in range(n)]
        assert any(r["status"] == 5 for r in refs) or thr == 0.3
        for cap in (mi + 2, mi + 7, 3 * (mi + 2)):
            rh = ctx.planner_batch(maps, se, prob_map=pmap, threshold=thr, max_iter=mi, ls_cap=cap)
            rd = run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=thr, max_iter=mi, ls_cap=cap)
            assert rh["light_sources"].shape == rd["light_sources"].shape == (n, cap, 2)
            for k in range(n):
                check(rh, k, refs[k])
                check(rd, k, refs[k])


def test_ls_cap_and_max_iter_rejected(ctx, vhp, torch):
    occ = np.ones((20, 30))
    se = [(1, 1, 25, 15)]
    for mi, cap in ((10, 11), (10, 0), (-1, 1), (-1, 5)):
        with pytest.raises(vhp.VhpError) as e:
            ctx.planner_batch(occ, se, threshold=0.5, max_iter=mi, ls_cap=cap)
        assert e.value.status == -1
        with pytest.raises(vhp.VhpError) as e:
            run_dev(ctx, vhp, torch, occ, se, thr=0.5, max_iter=mi, ls_cap=cap, which=SMALL if cap > 0 else ())
        assert e.value.status == -1
    # the context still works
    r = run_dev(ctx, vhp, torch, occ, se, thr=0.5, max_iter=10)
    assert int(r["status"][0]) == 0


# ---- degenerate problems ------------------------------------------------------------------------------
def test_degenerate_problems(ctx, vhp, torch, oracle):
    """1x1, 1xn, nx1 and 2x2 maps; start == end; start and end adjacent; the end walled off;
    thresholds 0, 1 and 1.5; both forms.

    Above 1 no cell reaches the threshold, so no cell is pushed and the reference takes the top of an
    empty heap, which is undefined.  The oracle then takes (0, 0) as the next source; the kernels stay
    on the source (the fixed point).  There only status, nb_sources, the start, the path and its
    length are compared."""
    walled = np.ones((9, 11))
    walled[2:7, 5] = walled[2, 5:10] = walled[6, 5:10] = walled[2:7, 9] = 0  # a closed box around (7, 4)
    cases = [(np.ones((1, 1)), [(0, 0, 0, 0)]),
             (np.ones((1, 9)), [(0, 0, 8, 0), (3, 0, 3, 0), (4, 0, 5, 0)]),
             (np.ones((9, 1)), [(0, 8, 0, 0), (0, 2, 0, 3)]),
             (np.ones((2, 2)), [(0, 0, 1, 1), (0, 0, 1, 0), (1, 1, 1, 1)]),
             (np.array([[1, 0], [0, 1]]), [(0, 0, 1, 1)]),
             (walled, [(1, 1, 7, 4), (7, 4, 7, 4), (7, 4, 1, 1)])]
    for occ, se in cases:
        for thr in (0.0, 1.0, 1.5):
            rh = ctx.planner_batch(occ, se, threshold=thr, max_iter=6)
            rd = run_dev(ctx, vhp, torch, occ, se, thr=thr, max_iter=6)
            for k in range(len(se)):
                ref = oracle.solve(occ.astype(np.float64), se[k][:2], se[k][2:], thr, 6)
                for r in (rh, rd):
                    if thr <= 1.0:
                        check(r, k, ref)
                        continue
                    assert (int(r["status"][k]), int(r["nb_sources"][k])) == (ref["status"], ref["nb_of_sources"])
                    if ref["status"] == 5:
                        assert tuple(r["light_sources"][k][0]) == tuple(se[k][:2])
                    assert int(r["path_n"][k]) == 0 and r["path_len"][k] == ref["path_length"] == 0.0


# ---- the bench's device leg ---------------------------------------------------------------------------
def bench_module():
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
    import bench
    return bench


def test_bench_device_leg(vhp, torch, oracle):
    """bench.py's device leg as it runs there: planner_workload(0), prepare_maps_dev, the device call
    with the six small outputs.  Every problem equals the host form, two per map equal the oracle.  Then
    the maps are regenerated into the same buffer (which drops the prepared planes) and overwritten
    from torch and prepared again: the results follow the buffer's content each time.  (The host form
    runs on a second context: a host call drops the planes its context prepared.)"""
    maps, se, pmap = bench_module().planner_workload(0)
    nmaps, ny, nx = maps.shape
    thr, mi = 0.5, 100
    c, h = make_ctx(vhp, torch), make_ctx(vhp, torch)
    with torch.cuda.stream(c.stream):
        occ_t = torch.from_numpy(maps).cuda()
    c.prepare_maps_dev(occ_t)

    def step(expect_maps, picks):
        rd = run_dev(c, vhp, torch, None, se, pmap=pmap, thr=thr, max_iter=mi, which=SMALL, occ_t=occ_t)
        rh = h.planner_batch(expect_maps, se, prob_map=pmap, threshold=thr, max_iter=mi, fields=False)
        same_results(rh, rd, SMALL, len(se))
        for k in picks:
            check(rd, k, oracle.solve(expect_maps[pmap[k]].astype(np.float64), se[k][:2], se[k][2:], thr, mi),
                  full=False)
        return rd

    per = len(se) // nmaps
    r0 = step(maps, [m * per + j for m in range(nmaps) for j in (0, 77)])
    assert (r0["status"] == 0).any() and (r0["status"] == 5).any()
    # regenerate into the same buffer: the planes prepared for the old content must not be used
    c.generate_environments_dev(occ_t, 12, 8, 40, 8, 40, 2024)
    c.stream.synchronize()
    new = occ_t.cpu().numpy()
    assert not np.array_equal(new, maps)
    r1 = step(new, range(0, len(se), 1024))
    assert not all(np.array_equal(r0[k], r1[k]) for k in ("status", "path_len"))
    # overwrite from torch, then prepare again
    flipped = np.ascontiguousarray(maps[:, ::-1, :])
    with torch.cuda.stream(c.stream):
        occ_t.copy_(torch.from_numpy(flipped).cuda())
    c.prepare_maps_dev(occ_t)
    step(flipped, range(5, len(se), 1024))
    c.close()
    h.close()


# ---- chunk edges --------------------------------------------------------------------------------------
def shipped_problems(oracle, n, seeds, rng):
    """n distinct problems over the shipped 1000^2 environments of `seeds` (prob_map cycles over them)."""
    maps = np.stack([oracle.generate_environment(1000, 1000, 15, 100, 200, 100, 200, s) for s in seeds])
    pmap = (np.arange(n) % len(seeds)).astype(np.int32)
    se = np.zeros((n, 4), np.int32)
    for m in range(len(seeds)):
        sel = np.flatnonzero(pmap == m)
        xs, ys = free_points(maps[m], 2 * len(sel), rng)
        se[sel] = np.stack([xs[: len(sel)], ys[: len(sel)], xs[len(sel):], ys[len(sel):]], axis=1)
    return maps, se, pmap


def test_host_staging_chunk_edge(vhp, torch, oracle):
    """The host form stages its outputs in 2 GiB chunks: 1000^2 maps with fp64 fields hold 107 problems
    per chunk.  115 problems on 6 maps equal the same problems run as batches below the edge; the
    problems on both sides of the edge and the last one equal the oracle."""
    per_chunk = (2 << 30) // (20 * 10**6 + 4 + 4 + 8 + 4 + 2 * 6 * 8 + 64)
    assert per_chunk == 107
    n, mi, thr = 115, 4, 0.25
    maps, se, pmap = shipped_problems(oracle, n, (1, 2, 3, 4, 5, 25), np.random.default_rng(115))
    c = make_ctx(vhp, torch)
    full = c.planner_batch(maps, se, prob_map=pmap, threshold=thr, max_iter=mi)
    for a, b in ((0, 100), (100, n)):
        part = c.planner_batch(maps, se[a:b], prob_map=pmap[a:b], threshold=thr, max_iter=mi)
        same_results({k: v[a:b] for k, v in full.items()}, part, ALL, b - a)
        del part
    c.close()
    for k in (per_chunk - 1, per_chunk, n - 1):
        check(full, k, oracle.solve(maps[pmap[k]], se[k][:2], se[k][2:], thr, mi))


def test_workspace_chunk_edge(vhp, torch, oracle):
    """planner_dev keeps the fields nobody asked for in a workspace of at most 32 GiB: 28 bytes per
    cell, so 1227 problems of 1000^2 per chunk.  1300 problems on 7 maps, in both forms: the first
    chunk takes the batch-wide first sweep (>= 8 x SMs problems), the second (73 problems) does not.
    Every problem equals the same problems run as two batches below the edge; the problems on both
    sides of the edge and the last one equal the oracle."""
    per_chunk = (32 << 30) // (28 * 10**6)
    assert per_chunk == 1227
    n, mi, thr = 1300, 4, 0.25
    maps, se, pmap = shipped_problems(oracle, n, (1, 2, 3, 4, 5, 6, 25), np.random.default_rng(1300))
    c = make_ctx(vhp, torch)
    with torch.cuda.stream(c.stream):
        occ_t = torch.from_numpy(np.ascontiguousarray(maps != 0, np.uint8)).cuda()
    rd = run_dev(c, vhp, torch, None, se, pmap=pmap, thr=thr, max_iter=mi, which=SMALL, occ_t=occ_t)
    rh = c.planner_batch(maps, se, prob_map=pmap, threshold=thr, max_iter=mi, fields=False)
    same_results(rd, rh, SMALL, n)
    for a, b in ((0, 650), (650, n)):
        part = run_dev(c, vhp, torch, None, se[a:b], pmap=pmap[a:b], thr=thr, max_iter=mi, which=SMALL, occ_t=occ_t)
        same_results({k: v[a:b] for k, v in rd.items()}, part, SMALL, b - a)
    c.close()
    assert len(set(map(tuple, rd["light_sources"][:, 1]))) > n // 2  # distinct problems
    for k in (per_chunk - 1, per_chunk, n - 1):
        check(rd, k, oracle.solve(maps[pmap[k]], se[k][:2], se[k][2:], thr, mi), full=False)


# ---- loop modes of the grid route ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def grid(vhp, torch):
    c = make_ctx(vhp, torch, "grid")
    yield c
    c.close()


def test_loop_modes(grid, vhp, oracle):
    """set_planner_loop 0 (automatic: the graph), 1 (graph), 2 (batches of 4 iterations), 3 (one read-back
    per iteration) on maze_5 and the shipped 1000^2 seed 1."""
    g, occ, se = maze5()
    ship = oracle.generate_environment(1000, 1000, 15, 100, 200, 100, 200, 1)
    ref = oracle.solve(ship, (50, 50), (990, 990), 0.25, 250)
    for mode in (0, 1, 2, 3):
        grid.set_planner_loop(mode)
        for tag, thr in (("thr020", 0.2), ("thr025", 0.25)):
            check_maze(grid.planner_batch(occ, [se], threshold=thr, max_iter=250), 0, g, tag)
        check(grid.planner_batch(ship, [(50, 50, 990, 990)], threshold=0.25, max_iter=250), 0, ref)
    grid.set_planner_loop(0)


def test_loop_mode2_batch_edges(grid, vhp, oracle):
    """Mode 2 enqueues 4 iterations per snapshot: max_iter 0..9 ends the loop inside a batch and exactly
    at its end, for a problem that runs into max_iter and for one that solves."""
    g, occ, se = maze5()
    rng = np.random.default_rng(9)
    xs, ys = free_points(occ, 2, rng)
    probs = [se, (int(xs[0]), int(ys[0]), int(xs[1]), int(ys[1]))]
    grid.set_planner_loop(2)
    try:
        for mi in range(10):
            for p in probs:
                ref = oracle.solve(occ.astype(np.float64), p[:2], p[2:], 0.25, mi)
                check(grid.planner_batch(occ, [p], threshold=0.25, max_iter=mi), 0, ref)
    finally:
        grid.set_planner_loop(0)


def test_loop_modes_switch_and_cached_engine(grid, vhp, oracle):
    """Modes switched back and forth on one context, and repeated solves on the cached engine with a
    different threshold, end point and map of the same shape."""
    g, occ, se = maze5()
    for mode in (1, 2, 3, 2, 1, 0, 3, 1):
        grid.set_planner_loop(mode)
        check_maze(grid.planner_batch(occ, [se], threshold=0.2, max_iter=250), 0, g, "thr020")
    grid.set_planner_loop(0)
    other = occ.copy()
    other[100:140, 60:200] = 0
    other[se[1], se[0]] = other[se[3], se[2]] = 1
    for mode in (1, 2):
        grid.set_planner_loop(mode)
        for m, p, thr in ((occ, se, 0.3), (occ, se, 0.2), (occ, (se[0], se[1], 30, 200), 0.2), (other, se, 0.2),
                          (other, se, 0.3), (occ, se, 0.3)):
            m = np.array(m)
            m[p[3], p[2]] = 1
            check(grid.planner_batch(m, [p], threshold=thr, max_iter=120), 0,
                  oracle.solve(m.astype(np.float64), p[:2], p[2:], thr, 120))
    grid.set_planner_loop(0)


def test_grid_route_device_prob_map(grid, vhp, torch, oracle):
    """Several problems on the grid route with a device prob_map (read back by the host); an index out
    of range is refused with VHP_ERR_INVALID_ARG."""
    nx, ny = 300, 260
    maps = np.stack([rect_map(nx, ny, 30, 300 + m, 5, 40) for m in range(3)])
    rng = np.random.default_rng(3)
    pmap = np.array([2, 0, 1, 2, 0], np.int32)
    se = np.zeros((5, 4), np.int32)
    for k in range(5):
        xs, ys = free_points(maps[pmap[k]], 2, rng)
        se[k] = (xs[0], ys[0], xs[1], ys[1])
    for dtype in (vhp.F64, vhp.F32):
        r = run_dev(grid, vhp, torch, maps, se, pmap=pmap, thr=0.3, max_iter=15, dtype=dtype)
        for k in range(5):
            check(r, k, oracle.solve(maps[pmap[k]], se[k][:2], se[k][2:], 0.3, 15), f32=dtype == vhp.F32)
    for bad in (3, -1):
        with pytest.raises(vhp.VhpError) as e:
            run_dev(grid, vhp, torch, maps, se, pmap=np.array([0, 1, bad, 2, 0], np.int32), thr=0.3, max_iter=15,
                    which=SMALL)
        assert e.value.status == -1


def test_loop_mode_rejected(grid, vhp):
    for mode in (4, -1):
        with pytest.raises(vhp.VhpError) as e:
            grid.set_planner_loop(mode)
        assert e.value.status == -1


# ---- the captured graph after the context's ratio table grows ----------------------------------------
def test_graph_recaptured_when_ratio_table_grows(vhp, torch, oracle):
    """The graph of the grid route's loop holds the context's reciprocal table, which a call on a
    larger map (side above 4040) or selftest_ratio(16384) frees and allocates again, larger.  A solve
    after that must use the new table."""
    g, occ, se = maze5()
    c = make_ctx(vhp, torch, "grid")
    check_maze(c.planner_batch(occ, [se], threshold=0.2, max_iter=250), 0, g, "thr020")
    wide = np.ones((8, 4200))
    wide[3, 1000:1010] = 0
    vis = c.visibility_batch(wide, [(5, 2)])
    assert np.array_equal(vis[0], oracle.compute_visibility(wide, 5, 2))
    check_maze(c.planner_batch(occ, [se], threshold=0.2, max_iter=250), 0, g, "thr020")
    assert c.selftest_ratio(16384) == 0
    check_maze(c.planner_batch(occ, [se], threshold=0.2, max_iter=250), 0, g, "thr020")
    c.close()


def test_giant_handle_graph_after_ratio_table_grows(vhp, torch):
    from visibility_heuristic_path_planner_b200.giant import GiantPlanner
    g, occ, se = maze5()
    c = make_ctx(vhp, torch)
    gp = GiantPlanner(occ, ctx=c)
    for step in range(2):
        r = gp.solve(se[:2], se[2:], 0.2, 250)
        assert r["stats"]["loop_mode"] == 1  # the graph
        assert (r["status"], r["nb_of_sources"]) == tuple(g["thr020_status"])
        assert np.array_equal(r["light_sources"], g["thr020_ls"]) and np.array_equal(r["path"], g["thr020_path"])
        assert r["path_length"] == g["thr020_len"][0]
        assert [sha(r["vg"]), sha(came_u64(r["came"])), sha(r["vis"])] == list(g["thr020_sha"])
        if step == 0:
            assert c.selftest_ratio(16384) == 0
    gp.close()
    c.close()


def test_grid_sweep_mode_change_on_cached_engine(vhp, torch, oracle):
    """set_grid_sweep 2 -> 1 -> 2 between solves of the same problem on one engine: the graph captured
    with one CTA count is not reused for the other, and every solve is exact."""
    ship = oracle.generate_environment(1000, 1000, 15, 100, 200, 100, 200, 1)
    ref = oracle.solve(ship, (50, 50), (990, 990), 0.25, 250)
    c = make_ctx(vhp, torch, "grid")
    for mode in (2, 1, 2, 1):
        c.set_grid_sweep(mode)
        check(c.planner_batch(ship, [(50, 50, 990, 990)], threshold=0.25, max_iter=250), 0, ref)
    c.close()
