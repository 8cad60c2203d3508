"""Merged visibility of groups of light sources (vhp_visibility_merge_batch) on the GPU: every route (the sweep
folding straight into the group outputs with 8-, 4- and 1-warp CTAs; grid mode, the naive kernel and thr <= 0
through the fp64 field and the fold kernel) against the oracle, against the library's own fields and against the
planner's visibility_global_ / cameFrom_.  All comparisons exact, fp64 and fp32."""
import numpy as np
import pytest

from conftest import load_golden, rect_map
from test_merge_cpu import came_u64, fold_fields, sha

pytestmark = pytest.mark.gpu
THRS = (0.5, 1.0, 1e-9, 0.9999999999, 0.0, -1.0)


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def make_groups(rng, nx, ny, occ, sizes):
    """Sources per group: corners, edges, x on word boundaries (x mod 32 in {0, 31}), occupied cells and
    duplicates first, random cells after."""
    special = [(0, 0), (nx - 1, ny - 1), (0, ny - 1), (nx - 1, 0), (min(31, nx - 1), ny // 2), (min(32, nx - 1), 0),
               (min(63, nx - 1), ny - 1), (nx // 2, 0), (0, ny // 2)]
    occd = np.argwhere(occ == 0)
    if len(occd):
        special += [(int(x), int(y)) for y, x in occd[:2]]
    special.append(special[0])  # duplicate
    srcs = []
    for gi, n in enumerate(sizes):
        g = [special[(gi + i) % len(special)] if i < len(special) else
             (int(rng.integers(0, nx)), int(rng.integers(0, ny))) for i in range(n)]
        if n >= 2:
            g[-1] = g[0]  # a duplicate inside the group
        srcs += g
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return np.array(srcs, np.int32).reshape(-1, 2), ptr


def expected(fields, srcs, ptr, thr, shape):
    outs = [fold_fields(fields[ptr[g]:ptr[g + 1]], srcs[ptr[g]:ptr[g + 1]], thr, shape) for g in range(len(ptr) - 1)]
    return [np.stack([o[i] for o in outs]) if outs else None for i in range(3)]


def check(r, want, dtype_f32, what):
    vmax, first, count = want
    wv = vmax.astype(np.float32) if dtype_f32 else vmax
    assert np.array_equal(r["vmax"], wv), what
    assert np.array_equal(r["first"], first), what
    assert np.array_equal(r["count"], count), what


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle_fold(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    sizes = [0, 1, 2, 7, 33, 0, 2]
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 2 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr))
    fields = np.stack([oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)])
    for thr in THRS:
        want = expected(fields, srcs, ptr, thr, (ny, nx))
        for dt in (vhp.F64, vhp.F32):
            r = ctx.visibility_merge_batch(occ, srcs, ptr, thr, group_map=gmap, dtype=dt)
            check(r, want, dt == vhp.F32, (shape, thr, dt))


@pytest.mark.parametrize("n", [12, 400, 2500])  # 8-, 4- and 1-warp CTAs (tile_warps_for)
def test_direct_kernels_against_library_fields(vhp, n):
    rng = np.random.default_rng(n)
    c = vhp.Context(0)
    for nx, ny, nobs in ((101, 101, 10), (97, 130, 0), (33, 32, 1), (160, 45, 12)):
        occ = np.stack([rect_map(nx, ny, nobs, 90 + k, 3, 14) for k in range(3)])
        ngroups = 3 if n <= 12 else n // 20
        ptr = np.sort(np.concatenate([[0, n], rng.integers(0, n + 1, ngroups - 1)])).astype(np.int64)
        sizes = np.diff(ptr)
        nsrc = int(ptr[-1])
        srcs = np.stack([rng.integers(0, nx, nsrc), rng.integers(0, ny, nsrc)], 1).astype(np.int32)
        srcs[:4] = [(0, 0), (nx - 1, ny - 1), (31, 5), (32 % nx, 0)]
        gmap = rng.integers(0, 3, len(sizes)).astype(np.int32)
        pmap = np.repeat(gmap, sizes)
        fields = c.visibility_batch(occ, srcs, src_map=pmap, dtype=vhp.F64)
        for thr in (0.5, 1.0, 1e-9, 0.9999999999):
            want = expected(fields, srcs, ptr, thr, (ny, nx))
            for dt in (vhp.F64, vhp.F32):
                check(c.visibility_merge_batch(occ, srcs, ptr, thr, group_map=gmap, dtype=dt), want, dt == vhp.F32,
                      (n, nx, ny, thr, dt))
    c.close()


@pytest.mark.parametrize("nobs", [0, 60])
def test_direct_kernel_1000(vhp, oracle, nobs):
    """1000 x 1000 maps with obstacles (every tile kind, dark runs) and empty (all lit: only the staircase); 24 pairs
    take the one-CTA kernel (4 and fewer would take grid mode)."""
    rng = np.random.default_rng(nobs)
    c = vhp.Context(0)
    occ = np.stack([oracle.generate_environment(1000, 1000, nobs, 10, 100, 10, 100, 5 + m) if nobs
                    else np.ones((1000, 1000)) for m in range(2)])
    sizes = np.array([8, 1, 0, 15], np.int64)
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    srcs = np.stack([rng.integers(0, 1000, 24), rng.integers(0, 1000, 24)], 1).astype(np.int32)
    srcs[:3] = [(0, 0), (999, 999), (512, 0)]
    gmap = np.array([0, 1, 0, 1], np.int32)
    fields = c.visibility_batch(occ, srcs, src_map=np.repeat(gmap, sizes), dtype=vhp.F64)
    for thr in (0.5, 1.0, 1e-9):
        want = expected(fields, srcs, ptr, thr, (1000, 1000))
        for dt in (vhp.F64, vhp.F32):
            check(c.visibility_merge_batch(occ, srcs, ptr, thr, group_map=gmap, dtype=dt), want, dt == vhp.F32,
                  (nobs, thr, dt))
    c.close()


def test_planner_identity(ctx, vhp):
    """visibility_global_ and cameFrom_ of planner_batch equal the merge over each problem's light sources."""
    rng = np.random.default_rng(5)
    nx, ny = 90, 70
    occ = np.stack([rect_map(nx, ny, 14, 300 + m, 3, 12) for m in range(6)])
    occ[:, :4, :4] = 1
    for thr, max_iter in ((0.25, 100), (0.5, 100), (0.0, 100), (1.0, 100), (0.3, 2)):
        n = 8
        se = np.stack([rng.integers(0, 4, n), rng.integers(0, 4, n), rng.integers(0, nx, n), rng.integers(0, ny, n)], 1)
        pm = rng.integers(0, 6, n).astype(np.int32)
        r = ctx.planner_batch(occ, se.astype(np.int32), prob_map=pm, threshold=thr, max_iter=max_iter)
        keep = [q for q in range(n) if int(r["status"][q]) in (0, 5)]
        assert keep
        nb = np.array([int(r["nb_sources"][q]) for q in keep], np.int64)
        srcs = np.concatenate([r["light_sources"][q][: nb[i]] for i, q in enumerate(keep)]).astype(np.int32)
        ptr = np.concatenate([[0], np.cumsum(nb)]).astype(np.int64)
        m = ctx.visibility_merge_batch(occ, srcs, ptr, thr, group_map=pm[keep], outputs=("vmax", "first"))
        for i, q in enumerate(keep):
            assert np.array_equal(m["vmax"][i], r["vg"][q]), (thr, q)
            assert np.array_equal(m["first"][i], r["came"][q]), (thr, q)
        if max_iter == 2:
            assert any(int(r["status"][q]) == 5 for q in keep)  # stalls to max_iter


def test_planner_identity_maze5(ctx, vhp):
    g = load_golden("maze5.npz")
    ny, nx = g["shape"]
    occ = np.unpackbits(g["occ_bits"])[: ny * nx].reshape(ny, nx)
    for tag, thr in (("thr020", 0.2), ("thr025", 0.25)):
        st, nb = g[f"{tag}_status"]
        ls = g[f"{tag}_ls"][:nb]
        r = ctx.visibility_merge_batch(occ, ls, [0, nb], thr, outputs=("vmax", "first"))
        assert [sha(r["vmax"][0]), sha(came_u64(r["first"][0]))] == list(g[f"{tag}_sha"][:2]), tag


def test_routes_agree(vhp, monkeypatch):
    rng = np.random.default_rng(11)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 12, 40 + m, 3, 14) for m in range(2)])
    srcs, ptr = make_groups(rng, nx, ny, occ[0], [5, 0, 12, 1, 30])
    gmap = np.array([1, 0, 0, 1, 1], np.int32)
    direct = vhp.Context(0)
    grid = vhp.Context(0)
    grid.set_grid_sweep(2)
    monkeypatch.setenv("VHP_SWEEP_IMPL", "naive")
    naive = vhp.Context(0)
    monkeypatch.delenv("VHP_SWEEP_IMPL")
    for thr in (0.5, 1e-9, 0.0):
        for dt in (vhp.F64, vhp.F32):
            rs = [c.visibility_merge_batch(occ, srcs, ptr, thr, group_map=gmap, dtype=dt) for c in (direct, grid, naive)]
            for r in rs[1:]:
                for k in ("vmax", "first", "count"):
                    assert np.array_equal(r[k], rs[0][k]), (thr, dt, k)
    for c in (direct, grid, naive):
        c.close()


def test_dev_equals_host(vhp):
    import torch
    rng = np.random.default_rng(3)
    nx, ny = 130, 96
    occ = np.stack([rect_map(nx, ny, 15, 60 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    srcs, ptr = make_groups(rng, nx, ny, occ[2], [4, 9, 0, 1, 40, 3])
    gmap = np.array([2, 0, 1, 2, 1, 0], np.int32)
    stream = torch.cuda.Stream()
    c = vhp.torch_context(0, stream)
    d = torch.device("cuda:0")
    occ_t = torch.from_numpy(occ).to(d)
    xy_t = torch.from_numpy(srcs).to(d)
    ptr_t = torch.from_numpy(ptr).to(d)
    gm_t = torch.from_numpy(gmap).to(d)
    ng = len(ptr) - 1
    for thr in (0.5, 0.0):
        for dt, tdt in ((vhp.F64, torch.float64), (vhp.F32, torch.float32)):
            host = c.visibility_merge_batch(occ, srcs, ptr, thr, group_map=gmap, dtype=dt)
            with torch.cuda.stream(stream):
                vm = torch.full((ng, ny, nx), 7.0, dtype=tdt, device=d)  # the call overwrites every cell
                fi = torch.full((ng, ny, nx), 5, dtype=torch.int32, device=d)
                co = torch.full((ng, ny, nx), 5, dtype=torch.int32, device=d)
                c.visibility_merge_batch_dev(occ_t, xy_t, ptr_t, thr, vmax_t=vm, first_t=fi, count_t=co, group_map_t=gm_t)
            c.synchronize()
            assert np.array_equal(vm.cpu().numpy(), host["vmax"])
            assert np.array_equal(fi.cpu().numpy(), host["first"])
            assert np.array_equal(co.cpu().numpy().view(np.uint32), host["count"])
    c.close()


def test_errors(vhp):
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    srcs = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    bad = [
        dict(src_xy=np.array([(1, 1), (30, 5), (7, 2)], np.int32), group_ptr=[0, 3]),  # source outside
        dict(group_ptr=[0, 1, 3], group_map=[0, 1]),                                     # map out of range
        dict(group_ptr=[0, 1, 3], group_map=[0, -1]),
        dict(group_ptr=[1, 3]),                                                          # does not start at 0
        dict(group_ptr=[0, 2, 1, 3]),                                                    # decreasing
        dict(group_ptr=[0, 2**31]),                                                      # group of 2^31 sources
        dict(group_ptr=[0, 3], threshold=float("nan")),
        dict(group_ptr=[0, 3], outputs=()),
    ]
    for b in bad:
        kw = dict(src_xy=srcs, threshold=0.5)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_merge_batch(occ, kw.pop("src_xy"), kw.pop("group_ptr"), kw.pop("threshold"), **kw)
        assert e.value.status == -1, b
        r = c.visibility_merge_batch(occ, srcs, [0, 3], 0.5)  # the context still works
        assert r["count"][0].max() == 3
    # empty groups and no groups are legal
    r = c.visibility_merge_batch(occ, srcs, [0, 0, 3, 3], 0.5)
    assert r["count"].shape == (3, 20, 30) and not r["count"][0].any() and (r["first"][2] == -1).all()
    assert r["vmax"].shape == (3, 20, 30) and not r["vmax"][[0, 2]].any()
    assert c.visibility_merge_batch(occ, np.zeros((0, 2), np.int32), [0], 0.5)["vmax"].shape == (0, 20, 30)
    # the _dev form reports a bad source / group layout through the device error flag
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    vm = torch.empty((2, 20, 30), dtype=torch.float64, device=d)
    for xy, ptr in (([(1, 1), (31, 1), (2, 2)], [0, 1, 3]), ([(1, 1), (3, 1), (2, 2)], [0, 2, 1]),
                    ([(1, 1), (3, 1), (2, 2)], [0, 1, 2])):
        c.visibility_merge_batch_dev(occ_t, torch.tensor(xy, dtype=torch.int32, device=d),
                                     torch.tensor(ptr, dtype=torch.int64, device=d), 0.5, vmax_t=vm)
        with pytest.raises(vhp.VhpError) as e:
            c.synchronize()
        assert e.value.status == -1, (xy, ptr)
    c.visibility_merge_batch_dev(occ_t, torch.tensor([(1, 1), (3, 1), (2, 2)], dtype=torch.int32, device=d),
                                 torch.tensor([0, 1, 3], dtype=torch.int64, device=d), 0.5, vmax_t=vm)
    c.synchronize()
    assert (vm == 1.0).sum().item() > 0
    c.close()


def test_contention_one_group_4096_sources(vhp):
    """One group of 4096 sources on an empty 1000 x 1000 map: every source folds into the same 1000 x 1000
    outputs at once.  Against the chunked fold of the library's own fields."""
    import torch
    rng = np.random.default_rng(4096)
    nx = ny = 1000
    n = 4096
    srcs = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
    srcs[:4] = [(0, 0), (0, 500), (500, 0), (999, 999)]
    c = vhp.Context(0)
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, ny, nx), dtype=torch.uint8, device=d)
    xy_t = torch.from_numpy(srcs).to(d)
    thr = 0.5
    vmax = torch.zeros((ny, nx), dtype=torch.float64, device=d)
    count = torch.zeros((ny, nx), dtype=torch.int64, device=d)
    first = torch.full((ny, nx), -1, dtype=torch.int64, device=d)
    buf = torch.empty((256, ny, nx), dtype=torch.float64, device=d)
    for p0 in range(0, n, 256):
        c.visibility_batch_dev(occ_t, xy_t[p0:p0 + 256].contiguous(), buf)
        c.synchronize()
        hit = buf >= thr
        hit[xy_t[p0:p0 + 256, 0] != 0, :, 0] = False  # the never-written border of each sweep
        hit[xy_t[p0:p0 + 256, 1] != 0, 0, :] = False
        count += hit.sum(0)
        new = (first < 0) & hit.any(0)
        first[new] = p0 + torch.argmax(hit.to(torch.uint8), 0)[new]
        vmax = torch.maximum(vmax, buf.max(0).values)
    r = c.visibility_merge_batch(np.ones((ny, nx)), srcs, [0, n], thr)
    assert np.array_equal(r["vmax"][0], vmax.cpu().numpy())
    assert np.array_equal(r["count"][0].astype(np.int64), count.cpu().numpy())
    assert np.array_equal(r["first"][0].astype(np.int64), first.cpu().numpy())
    c.close()
