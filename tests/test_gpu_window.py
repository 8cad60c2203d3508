"""Range-limited visibility (vhp_visibility_window_batch) on the GPU: the windowed tile kernel with 8-, 4- and 1-warp
CTAs, and the fallback through full fields (grid mode, the naive kernel), against the oracle, against crops of the
library's own full fields (also beyond the one-CTA kernel's map limit), against each other, and for stores that
stay inside each pair's window.  All comparisons exact, fp64 and fp32."""
import numpy as np
import pytest

from conftest import rect_map
from test_window_cpu import window_of

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(vhp):
    c = vhp.Context(0)
    yield c
    c.close()


def special_sources(nx, ny, occ):
    """corners, edges, x mod 32 in {0, 31}, occupied cells and a duplicate"""
    s = [(0, 0), (nx - 1, ny - 1), (0, ny - 1), (nx - 1, 0), (min(31, nx - 1), ny // 2), (min(32, nx - 1), 0),
         (min(63, nx - 1), ny - 1), (nx // 2, 0), (0, ny // 2)]
    occd = np.argwhere(occ == 0)
    s += [(int(x), int(y)) for y, x in occd[:2]]
    s.append(s[0])
    return s


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (29, 1), (40, 33), (64, 50), (160, 45)])
def test_oracle(ctx, vhp, oracle, shape):
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny)
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 400), 7 + m, 1, 6) for m in range(2)])
    srcs = special_sources(nx, ny, occ[1])
    srcs += [(int(rng.integers(0, nx)), int(rng.integers(0, ny))) for _ in range(6)]
    srcs = np.array(srcs, np.int32)
    pmap = (np.arange(len(srcs)) % 2).astype(np.int32)
    fields = [oracle.compute_visibility(occ[m], int(sx), int(sy)) for (sx, sy), m in zip(srcs, pmap)]
    for R in (0, 1, 5, 31, 32, 33, 100, max(nx, ny) + 3):
        want = np.stack([window_of(f, int(sx), int(sy), R) for f, (sx, sy) in zip(fields, srcs)])
        for dt in (vhp.F64, vhp.F32):
            got = ctx.visibility_window_batch(occ, srcs, R, src_map=pmap, dtype=dt)
            assert np.array_equal(got, want.astype(np.float32) if dt == vhp.F32 else want), (shape, R, dt)


def crops_of_fields(c, torch, occ_t, xy, pmap, R, chunk=64):
    """windows cut out of the library's full fp64 fields (visibility_batch_dev, `chunk` fields at a time)"""
    nmaps, ny, nx = occ_t.shape
    n = xy.shape[0]
    d = occ_t.device
    out = torch.empty((n, 2 * R + 1, 2 * R + 1), dtype=torch.float64, device=d)
    buf = torch.empty((min(chunk, n), ny, nx), dtype=torch.float64, device=d)
    for p0 in range(0, n, chunk):
        np_ = min(chunk, n - p0)
        torch.cuda.synchronize()  # torch is done with buf (the context has a stream of its own)
        c.visibility_batch_dev(occ_t, xy[p0:p0 + np_].contiguous(), buf[:np_],
                               src_map_t=None if pmap is None else pmap[p0:p0 + np_].contiguous())
        c.synchronize()
        padded = torch.nn.functional.pad(buf[:np_], (R, R, R, R))
        h = xy[p0:p0 + np_].cpu().numpy()
        for k in range(np_):
            sx, sy = int(h[k, 0]), int(h[k, 1])
            out[p0 + k] = padded[k, sy:sy + 2 * R + 1, sx:sx + 2 * R + 1]
    torch.cuda.synchronize()
    return out


def differing_pairs(torch, got, want):
    return torch.nonzero((got != want).flatten(1).any(1)).flatten()[:8].tolist()


def obstacle_maps(torch, c, nmaps, nx, ny, nobs, seed):
    occ_t = torch.empty((nmaps, ny, nx), dtype=torch.uint8, device="cuda:0")
    c.generate_environments_dev(occ_t, nobs, 10, 100, 10, 100, seed)
    return occ_t


@pytest.mark.parametrize("R,n", [(16, 12), (16, 400), (16, 2500), (128, 12), (128, 400), (128, 2500),
                                 (500, 12), (500, 400)])  # windows of <= 512: 8-, 4- and 1-warp CTAs by n
def test_against_library_fields(vhp, R, n):
    import torch
    from bench import workload
    c = vhp.Context(0)
    rng = np.random.default_rng(R * 10000 + n)
    shipped = torch.from_numpy(np.ascontiguousarray(workload("c2s", 0)[0][:1], dtype=np.uint8)).cuda()  # the shipped 1000 x 1000 map
    for occ_t in (shipped, obstacle_maps(torch, c, 2, 2048, 300, 60, 17)):
        nmaps, ny, nx = occ_t.shape
        xy = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        xy[:6] = [(0, 0), (nx - 1, ny - 1), (0, ny - 1), (nx - 1, 0), (31, ny // 2), (32, 1)]
        xy_t = torch.from_numpy(xy).cuda()
        pm_t = torch.from_numpy(rng.integers(0, nmaps, n).astype(np.int32)).cuda() if nmaps > 1 else None
        want = crops_of_fields(c, torch, occ_t, xy_t, pm_t, R)
        w64 = torch.empty_like(want)
        w32 = torch.empty(want.shape, dtype=torch.float32, device=want.device)
        c.visibility_window_batch_dev(occ_t, xy_t, R, w64, src_map_t=pm_t)
        c.visibility_window_batch_dev(occ_t, xy_t, R, w32, src_map_t=pm_t)
        c.synchronize()
        assert bool(torch.equal(w64, want)), (nx, ny, R, n, differing_pairs(torch, w64, want))
        assert bool(torch.equal(w32, want.float())), (nx, ny, R, n, differing_pairs(torch, w32, want.float()))
    c.close()


def test_beyond_one_cta_map_limit(vhp):
    """12000 x 12000: too wide for the one-CTA kernel's whole-map state, a window of R = 256 is not"""
    import torch
    c = vhp.Context(0)
    occ_t = obstacle_maps(torch, c, 1, 12000, 12000, 8000, 3)
    xy = np.array([(0, 0), (11999, 11999), (6000, 6000), (31, 11999), (11968, 17), (5000, 256), (255, 7000)], np.int32)
    xy_t = torch.from_numpy(xy).cuda()
    R = 256
    want = crops_of_fields(c, torch, occ_t, xy_t, None, R, chunk=1)
    for tdt in (torch.float64, torch.float32):
        got = torch.empty(want.shape, dtype=tdt, device=want.device)
        c.visibility_window_batch_dev(occ_t, xy_t, R, got)
        c.synchronize()
        assert bool(torch.equal(got, want.to(tdt))), (tdt, differing_pairs(torch, got, want.to(tdt)))
    c.close()


def test_routes_agree(vhp, monkeypatch):
    rng = np.random.default_rng(11)
    nx, ny = 101, 77
    occ = np.stack([rect_map(nx, ny, 12, 40 + m, 3, 14) for m in range(2)])
    srcs = np.array(special_sources(nx, ny, occ[0]) + [(int(rng.integers(0, nx)), int(rng.integers(0, ny)))
                                                       for _ in range(20)], np.int32)
    pmap = rng.integers(0, 2, len(srcs)).astype(np.int32)
    direct = vhp.Context(0)
    grid = vhp.Context(0)
    grid.set_grid_sweep(2)
    monkeypatch.setenv("VHP_SWEEP_IMPL", "naive")
    naive = vhp.Context(0)
    monkeypatch.delenv("VHP_SWEEP_IMPL")
    for R in (0, 7, 40, 200):
        for dt in (vhp.F64, vhp.F32):
            rs = [c.visibility_window_batch(occ, srcs, R, src_map=pmap, dtype=dt) for c in (direct, grid, naive)]
            for r in rs[1:]:
                assert np.array_equal(r, rs[0]), (R, dt)
    for c in (direct, grid, naive):
        c.close()


@pytest.mark.parametrize("n", [12, 2500])
def test_no_stray_stores(vhp, n):
    """The windows are a view into a NaN-filled tensor with margins before the first and after the last; sources at
    all four corners (three quarters of those windows lie outside the grid).  The margins keep their NaN bits, the
    out-of-grid cells are 0, the rest is the host form's result."""
    import torch
    rng = np.random.default_rng(n)
    nx, ny, R = 100, 70, 20
    occ = rect_map(nx, ny, 15, 5, 3, 10)
    xy = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
    xy[:4] = [(0, 0), (nx - 1, 0), (0, ny - 1), (nx - 1, ny - 1)]
    xy[-4:] = xy[:4]
    c = vhp.Context(0)
    occ_t = torch.from_numpy(occ.astype(np.uint8)[None]).cuda()
    xy_t = torch.from_numpy(xy).cuda()
    W, margin = 2 * R + 1, 777
    for tdt, dt in ((torch.float64, vhp.F64), (torch.float32, vhp.F32)):
        big = torch.full((2 * margin + n * W * W,), float("nan"), dtype=tdt, device="cuda:0")
        canary = big[:1].clone()
        out = big[margin:margin + n * W * W].view(n, W, W)
        torch.cuda.synchronize()  # the fill, before the context's stream writes
        c.visibility_window_batch_dev(occ_t, xy_t, R, out)
        c.synchronize()
        ib = torch.int64 if tdt == torch.float64 else torch.int32
        assert bool((big[:margin].view(ib) == canary.view(ib)).all()) and bool((big[-margin:].view(ib) == canary.view(ib)).all())
        host = c.visibility_window_batch(occ, xy, R, dtype=dt)
        assert np.array_equal(out.cpu().numpy(), host)
        xs = xy[:, 0, None] - R + np.arange(W)[None, :]
        ys = xy[:, 1, None] - R + np.arange(W)[None, :]
        outside = ~(((ys >= 0) & (ys < ny))[:, :, None] & ((xs >= 0) & (xs < nx))[:, None, :])
        assert outside[:4].sum() == 4 * (W * W - (R + 1) ** 2) and not host[outside].any()
    c.close()


def test_dev_equals_host_and_prepared_maps(vhp):
    import torch
    rng = np.random.default_rng(3)
    nx, ny = 130, 96
    occ = np.stack([rect_map(nx, ny, 15, 60 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    xy = np.array(special_sources(nx, ny, occ[2]) + [(int(rng.integers(0, nx)), int(rng.integers(0, ny)))
                                                     for _ in range(40)], np.int32)
    pm = rng.integers(0, 3, len(xy)).astype(np.int32)
    stream = torch.cuda.Stream()
    c = vhp.torch_context(0, stream)
    occ_t, xy_t, pm_t = (torch.from_numpy(a).cuda() for a in (occ, xy, pm))
    torch.cuda.synchronize()
    for R in (3, 50):
        for dt, tdt in ((vhp.F64, torch.float64), (vhp.F32, torch.float32)):
            host = c.visibility_window_batch(occ, xy, R, src_map=pm, dtype=dt)
            with torch.cuda.stream(stream):
                out = torch.full((len(xy), 2 * R + 1, 2 * R + 1), 7.0, dtype=tdt, device="cuda:0")
                c.visibility_window_batch_dev(occ_t, xy_t, R, out, src_map_t=pm_t)
            c.synchronize()
            assert np.array_equal(out.cpu().numpy(), host), (R, dt)
            with torch.cuda.stream(stream):  # the packed planes of vhp_prepare_maps_dev, used twice
                c.prepare_maps_dev(occ_t)
                again = [torch.full_like(out, 5.0) for _ in range(2)]
                for a in again:
                    c.visibility_window_batch_dev(occ_t, xy_t, R, a, src_map_t=pm_t)
            c.synchronize()
            for a in again:
                assert np.array_equal(a.cpu().numpy(), host), (R, dt)
    c.lib.vhp_release_maps_dev(c.h)
    c.close()


def test_errors(vhp, monkeypatch):
    import ctypes as C
    import torch
    c = vhp.Context(0)
    occ = np.ones((20, 30))
    xy = np.array([(1, 1), (5, 5), (7, 2)], np.int32)
    bad = [dict(radius=-1), dict(radius=16384), dict(src_xy=np.array([(1, 1), (30, 5)], np.int32)),
           dict(src_xy=np.array([(1, 1), (3, -1)], np.int32)), dict(src_map=np.array([0, 1, 0], np.int32)),
           dict(src_map=np.array([0, -1, 0], np.int32))]
    for b in bad:
        kw = dict(src_xy=xy, radius=4)
        kw.update(b)
        with pytest.raises(vhp.VhpError) as e:
            c.visibility_window_batch(occ, kw.pop("src_xy"), kw.pop("radius"), **kw)
        assert e.value.status == -1, b
        assert c.visibility_window_batch(occ, xy, 4)[0, 4, 4] == 1.0  # the context still works
    occ8 = np.ones((1, 20, 30), np.uint8)
    st = c.lib.vhp_visibility_window_batch(c.h, occ8.ctypes.data_as(C.c_void_p), 1, 30, 20,
                                           xy.ctypes.data_as(C.c_void_p), None, 3, 4, vhp.F64, None)
    assert st == -1  # null out
    assert c.visibility_window_batch(occ, np.zeros((0, 2), np.int32), 4).shape == (0, 9, 9)
    # the _dev form reports a bad source / map index through the device error flag, on every route
    d = torch.device("cuda:0")
    occ_t = torch.ones((1, 20, 30), dtype=torch.uint8, device=d)
    out = torch.empty((3, 9, 9), dtype=torch.float64, device=d)
    monkeypatch.setenv("VHP_SWEEP_IMPL", "naive")
    naive = vhp.Context(0)
    monkeypatch.delenv("VHP_SWEEP_IMPL")
    for cc in (c, naive):
        for pts, pm in (([(1, 1), (31, 1), (2, 2)], None), ([(1, 1), (3, 1), (2, 2)], [0, 1, 0])):
            cc.visibility_window_batch_dev(occ_t, torch.tensor(pts, dtype=torch.int32, device=d), 4, out,
                                           src_map_t=None if pm is None else torch.tensor(pm, dtype=torch.int32,
                                                                                          device=d))
            with pytest.raises(vhp.VhpError) as e:
                cc.synchronize()
            assert e.value.status == -1, (pts, pm)
        with pytest.raises(vhp.VhpError):
            cc.visibility_window_batch_dev(occ_t, torch.tensor(xy, device=d), 16384, out)
        cc.visibility_window_batch_dev(occ_t, torch.tensor(xy, device=d), 4, out)
        cc.synchronize()
        assert bool((out[:, 4, 4] == 1.0).all())
    naive.close()
    c.close()
