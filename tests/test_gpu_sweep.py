"""K1 (visibility sweep) and K4 (ray casting) on the GPU, through the C-ABI,
against the CPU oracle and the golden vectors.  Bit-exact in fp64; VHP_F32 output
must equal the oracle's fp64 value rounded once to fp32."""
import hashlib
import os

import numpy as np
import pytest

from conftest import load_golden, rect_map

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


# auto = the tile wavefront kernel, one CTA per pair; grid = the same tile body with every sweep
# spread over many CTAs (what a few sweeps of a large map take by default; forced here)
@pytest.fixture(scope="module", params=["auto", "naive", "grid"])
def ctx(request, vhp):
    os.environ["VHP_SWEEP_IMPL"] = "auto" if request.param == "grid" else request.param
    c = vhp.Context(0)
    os.environ.pop("VHP_SWEEP_IMPL")
    c.set_grid_sweep(2 if request.param == "grid" else 0)
    yield c
    c.close()


def oracle_batch(oracle, occ, srcs):
    return np.stack([oracle.compute_visibility(occ, sx, sy) for sx, sy in srcs])


def test_ratio_exact_exhaustive(vhp):
    c = vhp.Context(0)
    assert c.selftest_ratio(4096) == 0
    assert c.selftest_ratio(16384) == 0
    c.close()


def test_golden_sweeps(ctx, vhp):
    g = load_golden("sweep.npz")
    for k, (nx, ny, nobs, seed, sx, sy) in enumerate(g["cases"]):
        occ = g[f"occ_{k}"]
        out = ctx.visibility_batch(occ, [(sx, sy)], dtype=vhp.F64)[0]
        assert np.array_equal(out, g[f"vis_{k}"]), (k, nx, ny, sx, sy)
        out32 = ctx.visibility_batch(occ, [(sx, sy)], dtype=vhp.F32)[0]
        assert np.array_equal(out32, g[f"vis_{k}"].astype(np.float32)), k
    assert np.array_equal(ctx.visibility_batch(g["kat_diag_occ"], [(2, 2)])[0], g["kat_diag_vis"])
    occ = np.ones((12, 10)); occ[5, 4] = 0
    assert not ctx.visibility_batch(occ, [(4, 5)]).any()          # occupied source
    seed, x, y = map(int, g["kat_flip"])
    # strict-IEEE threshold decision (the -Ofast reference build flips this cell)
    from oracle_py import Oracle
    occ = Oracle().generate_environment(101, 101, 10, 10, 20, 10, 20, seed)
    out = ctx.visibility_batch(occ, [(50, 50)])[0]
    assert np.array_equal(out, g["kat_flip_vis"]) and out[y, x] == g["kat_flip_vals"][0]


@pytest.mark.parametrize("shape", [(1, 1), (1, 9), (9, 1), (2, 2), (3, 5), (31, 33), (64, 64),
                                   (127, 129), (130, 61), (257, 255), (256, 256), (300, 200),
                                   (513, 40), (40, 517), (12000, 40)])  # the last: too wide for the
                                                                        # one-CTA kernel (naive / grid only)
def test_random_maps_all_source_positions(ctx, vhp, oracle, shape):
    nx, ny = shape
    g = np.random.default_rng(nx * 1000 + ny)
    occ = rect_map(nx, ny, (nx * ny) // 400, nx + ny, 1, 9)
    srcs = [(0, 0), (nx - 1, 0), (0, ny - 1), (nx - 1, ny - 1), (nx // 2, ny // 2)]
    srcs += [(int(g.integers(0, nx)), int(g.integers(0, ny))) for _ in range(11)]
    ref = oracle_batch(oracle, occ, srcs)
    out = ctx.visibility_batch(occ, srcs, dtype=vhp.F64)
    bad = [(s, np.argwhere(o != r)[:3].tolist()) for s, o, r in zip(srcs, out, ref)
           if not np.array_equal(o, r)]
    assert not bad, bad[:3]
    out32 = ctx.visibility_batch(occ, srcs, dtype=vhp.F32)
    assert np.array_equal(out32, ref.astype(np.float32))


def test_multi_map_batch(ctx, vhp, oracle):
    nx, ny, nmaps = 96, 80, 7
    maps = np.stack([rect_map(nx, ny, 10, 50 + m, 2, 12) for m in range(nmaps)])
    g = np.random.default_rng(5)
    src_map = g.integers(0, nmaps, 40).astype(np.int32)
    srcs = np.stack([g.integers(0, nx, 40), g.integers(0, ny, 40)], axis=1).astype(np.int32)
    out = ctx.visibility_batch(maps, srcs, src_map=src_map)
    for p in range(40):
        assert np.array_equal(out[p], oracle.compute_visibility(maps[src_map[p]], *srcs[p])), p


def test_shipped_1000_config(ctx, vhp, oracle):
    """config/settings.config of the reference (1000x1000, 15 obstacles, seed 1)."""
    g = load_golden("shipped1000.npz")
    occ = oracle.generate_environment(1000, 1000, 15, 100, 200, 100, 200, 1)
    out = ctx.visibility_batch(occ, [(50, 50)], dtype=vhp.F64)[0]
    s64, s32, sbin = g["seed1_cv_sha"]
    assert sha(out) == s64
    assert sha((out >= 0.25).astype(np.uint8)) == sbin      # thresholded visibility bit-exact
    out32 = ctx.visibility_batch(occ, [(50, 50)], dtype=vhp.F32)[0]
    assert sha(out32) == s32
    empty = ctx.visibility_batch(np.ones((1000, 1000)), [(500, 500)])[0]
    assert sha(empty) == g["empty_cv_sha"][0]


def test_1000_random_sources_vs_oracle(ctx, vhp, oracle):
    occ = oracle.generate_environment(1000, 1000, 15, 100, 200, 100, 200, 3)
    g = np.random.default_rng(11)
    srcs = [(int(g.integers(0, 1000)), int(g.integers(0, 1000))) for _ in range(6)]
    srcs += [(0, 999), (999, 0), (3, 4), (996, 997)]
    out = ctx.visibility_batch(occ, srcs, dtype=vhp.F64)
    for s, o in zip(srcs, out):
        assert np.array_equal(o, oracle.compute_visibility(occ, *s)), s


def test_every_tile_alignment(vhp, oracle):
    """The first tile row / column of a quadrant is 1..32 cells wide depending on the
    source x: cover every residue of sx mod 32 (both store paths: fp64 / fp32, vector
    and scalar rows) on a map with obstacles and on an empty one."""
    c = vhp.Context(0)
    for nx, ny in ((200, 96), (197, 70)):
        occ = rect_map(nx, ny, 14, 4242 + nx, 3, 17)
        srcs = [(x, (7 * x + 3) % ny) for x in range(0, 70)] + [(nx - 1 - x, ny - 1) for x in range(0, 34)]
        ref = oracle_batch(oracle, occ, srcs)
        assert np.array_equal(c.visibility_batch(occ, srcs, dtype=vhp.F64), ref)
        assert np.array_equal(c.visibility_batch(occ, srcs, dtype=vhp.F32), ref.astype(np.float32))
        empty = np.ones((ny, nx))
        ref = oracle_batch(oracle, empty, srcs[:40])
        assert np.array_equal(c.visibility_batch(empty, srcs[:40], dtype=vhp.F32), ref.astype(np.float32))
    c.close()


def test_large_grid_vs_naive(vhp):
    """A grid beyond the BASELINE size (more than 32 x 32 tile columns per block-summary
    word row): tile kernel == naive kernel bit-for-bit."""
    from oracle_py import Oracle
    nx, ny = 2100, 1300
    occ = Oracle().generate_environment(nx, ny, 60, 20, 160, 20, 160, 5)
    srcs = [(0, 0), (nx - 1, ny - 1), (1050, 650), (2099, 3), (31, 1299), (1024, 1024)]
    os.environ["VHP_SWEEP_IMPL"] = "naive"
    a = vhp.Context(0)
    os.environ.pop("VHP_SWEEP_IMPL")
    b = vhp.Context(0)
    ra = a.visibility_batch(occ, srcs, dtype=vhp.F64)
    rb = b.visibility_batch(occ, srcs, dtype=vhp.F64)
    assert np.array_equal(ra, rb)
    a.close(); b.close()


def test_giant_grid_8192_vs_naive(vhp):
    """BASELINE configs[4] size (8192 x 8192 dense random obstacles): the tile kernel's
    boundary rows still fit shared memory (one CTA per SM); bit-identical to the naive
    kernel, fp32 store (fp64 on chip)."""
    n = 8192
    g = np.random.default_rng(8192)
    occ = np.ones((n, n), dtype=np.uint8)
    for _ in range(6000):
        x, y = int(g.integers(1, n)), int(g.integers(1, n))
        w, h = int(g.integers(8, 65)), int(g.integers(8, 65))
        occ[y:y + h, x:x + w] = 0
    srcs = [(int(x), int(y)) for y, x in np.argwhere(occ[4000:4100, 4000:4100] != 0)[:1] + 4000] + [(0, 0)]
    assert occ[srcs[0][1], srcs[0][0]] != 0
    os.environ["VHP_SWEEP_IMPL"] = "naive"
    a = vhp.Context(0)
    os.environ.pop("VHP_SWEEP_IMPL")
    b = vhp.Context(0)
    ra = a.visibility_batch(occ, srcs, dtype=vhp.F32)
    rb = b.visibility_batch(occ, srcs, dtype=vhp.F32)
    assert np.array_equal(ra, rb)
    assert int((rb[0] > 0.5).sum()) > 100 and float((rb[0] > 0.5).mean()) < 0.99
    a.close(); b.close()


def test_tile_equals_naive_full_size(vhp):
    """Size-independent property at BASELINE size: the tile kernel and the simple
    kernel agree bit-for-bit on a 64-source 1000x1000 batch."""
    from oracle_py import Oracle
    occ = Oracle().generate_environment(1000, 1000, 40, 20, 120, 20, 120, 9)
    g = np.random.default_rng(3)
    srcs = np.stack([g.integers(0, 1000, 64), g.integers(0, 1000, 64)], axis=1)
    os.environ["VHP_SWEEP_IMPL"] = "naive"
    a = vhp.Context(0)
    os.environ.pop("VHP_SWEEP_IMPL")
    b = vhp.Context(0)
    ra = a.visibility_batch(occ, srcs, dtype=vhp.F64)
    rb = b.visibility_batch(occ, srcs, dtype=vhp.F64)
    assert np.array_equal(ra, rb)
    assert ra.min() >= 0.0 and ra.max() <= 1.0
    a.close(); b.close()


def test_out_of_grid_source_is_an_error(ctx, vhp):
    with pytest.raises(vhp.VhpError) as e:
        ctx.visibility_batch(np.ones((8, 8)), [(8, 0)])
    assert e.value.status == -1


def test_raycast_vs_oracle(ctx, vhp, oracle):
    g = load_golden("sweep.npz")
    for k, (nx, ny, nobs, seed, sx, sy) in enumerate(g["cases"]):
        out = ctx.raycast_batch(g[f"occ_{k}"], [(sx, sy)], dtype=vhp.F64)[0]
        assert np.array_equal(out, g[f"ray_{k}"]), k
    occ = rect_map(200, 150, 40, 8, 3, 15)
    srcs = [(0, 0), (199, 149), (100, 75), (17, 140)]
    out = ctx.raycast_batch(occ, srcs, dtype=vhp.F32)
    for s, o in zip(srcs, out):
        assert np.array_equal(o, oracle.raycast_all(occ, *s).astype(np.float32)), s


def test_binary_visibility_bit_exact(ctx, vhp, oracle):
    """vhp_visibility_batch_bin: bit b of word w = (fp64 visibility >= threshold), bit-exact
    against the oracle's field for thresholds that occur exactly in the field (0.5, 1.0), the
    planner's defaults and the degenerate 0; several maps, odd widths, host and device entry."""
    import torch
    rng = np.random.default_rng(11)
    for nx, ny, nobs, seed in ((101, 101, 10, 7), (77, 133, 14, 3), (260, 40, 9, 5), (33, 31, 2, 1)):
        occ = np.stack([rect_map(nx, ny, nobs, seed + k, 3, 14) for k in range(3)])
        n = 12
        smap = rng.integers(0, 3, n).astype(np.int32)
        src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        src[0] = (nx // 2, ny // 2)
        ref = np.stack([oracle.compute_visibility(occ[m], sx, sy) for (sx, sy), m in zip(src, smap)])
        for thr in (0.5, 0.25, 1.0, 0.0, 1e-300, 0.49999999999999994):
            bits = ctx.visibility_batch_bin(occ, src, thr, src_map=smap)
            assert bits.shape == (n, ny, (nx + 31) // 32) and bits.dtype == np.uint32
            assert np.array_equal(vhp.unpack_bits(bits, nx), ref >= thr), (nx, ny, thr)
            pad = np.unpackbits(bits.view(np.uint8), axis=-1, bitorder="little")[..., nx:]
            assert not pad.any()  # bits beyond nx are 0
        dev = torch.device("cuda", 0)
        out_t = torch.full((n, ny, (nx + 31) // 32), -1, dtype=torch.int32, device=dev)
        ctx.visibility_batch_bin_dev(torch.from_numpy(occ != 0).to(torch.uint8).to(dev), torch.from_numpy(src).to(dev),
                                     0.5, out_t, torch.from_numpy(smap).to(dev))
        ctx.synchronize()
        assert np.array_equal(vhp.unpack_bits(out_t.cpu().numpy().view(np.uint32), nx), ref >= 0.5)
    # the strict-IEEE flip cell of SURVEY 8c: 0.49999999999999989 < 0.5 must read "not visible"
    g = load_golden("sweep.npz")
    seed, x, y = map(int, g["kat_flip"])
    occ = oracle.generate_environment(101, 101, 10, 10, 20, 10, 20, seed)
    bits = vhp.unpack_bits(ctx.visibility_batch_bin(occ, [(50, 50)], 0.5), 101)[0]
    assert not bits[y, x] and oracle.compute_visibility(occ, 50, 50)[y, x] < 0.5


def test_sweep_variants_equal_oracle(vhp, oracle):
    """vhp_visibility_variant_batch: getAccessibilityMap.m (alpha decay, fac curve factor) and the
    early-terminating computeVisibilityUsingQueue rule, bit-exact against their C restatements."""
    c = vhp.Context(0)
    rng = np.random.default_rng(21)
    for nx, ny, nobs, seed in ((64, 48, 12, 3), (101, 101, 25, 7), (33, 77, 8, 9), (260, 130, 40, 2)):
        occ = np.stack([rect_map(nx, ny, nobs, seed + k, 2, 11) for k in range(2)])
        n = 6
        smap = rng.integers(0, 2, n).astype(np.int32)
        src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        src[0] = (0, 0); src[1] = (nx - 1, ny - 1); src[2] = (nx // 2, 0)
        for alpha, fac, ls in ((1.0, 1.0, 1.0), (0.97, 1.0, 1.0), (1.0, 0.5, 1.0), (0.999, 2.0, 0.5), (1.0, 1.3, 1.0)):
            out = c.visibility_variant_batch(occ, src, vhp.VARIANT_MATLAB, alpha=alpha, fac=fac,
                                             light_strength=ls, src_map=smap)
            for k in range(n):
                ref = oracle.accessibility_map(occ[smap[k]], *src[k], alpha=alpha, fac=fac, light_strength=ls)
                assert np.array_equal(out[k], ref), (nx, ny, alpha, fac, k)
        for cutoff in (0.001, 0.0, 0.05):
            out = c.visibility_variant_batch(occ, src, vhp.VARIANT_QUEUE, cutoff=cutoff, src_map=smap)
            out32 = c.visibility_variant_batch(occ, src, vhp.VARIANT_QUEUE, cutoff=cutoff, src_map=smap, dtype=vhp.F32)
            for k in range(n):
                ref = oracle.visibility_cutoff(occ[smap[k]], *src[k], cutoff=cutoff)
                assert np.array_equal(out[k], ref), (nx, ny, cutoff, k)
                assert np.array_equal(out32[k], ref.astype(np.float32))
    # the reference's own output (golden fixture) where its queue order does not matter
    g = load_golden("queue.npz")
    done = 0
    for row in g["cases"][:40]:
        t, nx, ny, nobs, sx, sy = (int(v) for v in row[:6])
        if not g["agree"][t]:
            continue
        out = c.visibility_variant_batch(rect_map(nx, ny, nobs, t, 1, 9), [(sx, sy)], vhp.VARIANT_QUEUE)[0]
        assert np.array_equal(out, g[f"ref_{t}"]), t
        done += 1
    assert done >= 25
    with pytest.raises(vhp.VhpError):
        c.visibility_variant_batch(occ, src, 3)
    with pytest.raises(vhp.VhpError):
        c.visibility_variant_batch(occ, src, vhp.VARIANT_MATLAB, fac=0.0)
    c.close()


def test_binary_thresholds_on_field_values(vhp, oracle, monkeypatch):
    """The binary outputs come from sweeps that write bits themselves (csrc/sweep_tile_body.cuh
    kFmtBits, fp64 compare in the kernel): the bits must equal (fp64 value >= threshold) when the
    threshold IS a value of the field, its fp64 neighbours, its fp32 roundings and their neighbours
    -- where an fp32 round trip would flip -- and for thresholds <= 0, > 1, huge and denormal.  The
    fp64-field route (VHP_BIN_DIRECT=0: sweep, then threshold pass) gives the same bits."""
    rng = np.random.default_rng(23)
    nx, ny = 150, 117
    occ = np.stack([rect_map(nx, ny, 12, 40 + k, 3, 16) for k in range(2)])
    n = 6
    smap = rng.integers(0, 2, n).astype(np.int32)
    src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
    ref = np.stack([oracle.compute_visibility(occ[m], sx, sy) for (sx, sy), m in zip(src, smap)])
    vals = np.unique(ref[(ref > 0) & (ref < 1)])
    assert len(vals) > 100
    pick = rng.choice(vals, 12, replace=False)
    thrs = []
    for v in pick:
        f = np.float64(np.float32(v))
        thrs += [v, np.nextafter(v, 2.0), np.nextafter(v, -1.0), f,
                 np.float64(np.nextafter(np.float32(v), np.float32(2))),
                 np.float64(np.nextafter(np.float32(v), np.float32(-1)))]
    thrs += [-1.0, 2.0, -1e300, 1e300, np.inf, 1e-310, 5e-324]
    c = vhp.Context(0)
    monkeypatch.setenv("VHP_BIN_DIRECT", "0")
    c64 = vhp.Context(0)
    monkeypatch.delenv("VHP_BIN_DIRECT")
    for i, thr in enumerate(thrs):
        want = ref >= thr
        got = vhp.unpack_bits(c.visibility_batch_bin(occ, src, float(thr), src_map=smap), nx)
        assert np.array_equal(got, want), (i, thr)
        if i % 6 == 0:
            assert np.array_equal(vhp.unpack_bits(c64.visibility_batch_bin(occ, src, float(thr), src_map=smap), nx), want)
            rc, pp, tr = c.visibility_batch_runs(occ, src, float(thr), src_map=smap)
            assert np.array_equal(vhp.unpack_bits(vhp.runs_to_bits(rc, pp, tr, nx), nx), want)
    c.close(); c64.close()


@pytest.mark.parametrize("n", [400, 2500])  # 4-warp and single-warp CTAs (12 pairs above: 8 warps)
def test_binary_direct_all_warp_counts(vhp, n):
    """The bit-writing sweep at the batch sizes that select the 4-warp and the 1-warp kernels, with
    sources on word boundaries, corners and edges: equal to the fp64 field of the same library
    compared with >= threshold (the fields of those instances are checked against the oracle in
    test_gpu_warps.py, at these and other batch sizes)."""
    rng = np.random.default_rng(n)
    c = vhp.Context(0)
    for nx, ny, nobs in ((101, 101, 10), (64, 50, 5), (97, 130, 0), (33, 32, 1), (160, 45, 12)):
        occ = np.stack([rect_map(nx, ny, nobs, 90 + k, 3, 14) for k in range(4)])
        smap = rng.integers(0, 4, n).astype(np.int32)
        src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        special = [(0, 0), (nx - 1, ny - 1), (0, ny - 1), (nx - 1, 0), (31, 5), (32, 5), (33, 31), (63 % nx, 32 % ny),
                   (64 % nx, 0), (nx // 2, 0), (0, ny // 2), (nx - 1, ny // 2), (nx // 2, ny - 1)]
        src[: len(special)] = [(min(x, nx - 1), min(y, ny - 1)) for x, y in special]
        field = c.visibility_batch(occ, src, src_map=smap, dtype=vhp.F64)
        for thr in (0.5, 1.0, 1e-9, 0.9999999999):
            bits = c.visibility_batch_bin(occ, src, thr, src_map=smap)
            got = vhp.unpack_bits(bits, nx)
            bad = np.argwhere(got != (field >= thr))
            assert len(bad) == 0, (nx, ny, thr, bad[:5], src[bad[0][0]])
            assert not np.unpackbits(bits.view(np.uint8), axis=-1, bitorder="little")[..., nx:].any()
        rc, pp, tr = c.visibility_batch_runs(occ, src, 0.5, src_map=smap)
        assert np.array_equal(vhp.runs_to_bits(rc, pp, tr, nx), c.visibility_batch_bin(occ, src, 0.5, src_map=smap))
    c.close()


def test_binary_direct_large_maps(vhp):
    """Bit-writing sweeps of 1000 x 1000 and 1333 x 777 maps with many obstacles (dark runs, every tile
    kind) and of free maps (all lit), against the fp64 field; 3 pairs of the large map take the
    grid-mode route (fp64 field + threshold pass) and must agree too."""
    rng = np.random.default_rng(77)
    c = vhp.Context(0)
    for nx, ny, nobs, n in ((1000, 1000, 120, 24), (1333, 777, 60, 20), (1000, 1000, 0, 20), (1000, 1000, 40, 3)):
        occ = rect_map(nx, ny, nobs, 5, 10, 60)[None]
        src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        src[0] = (nx // 2, ny // 2)
        field = c.visibility_batch(occ, src, dtype=vhp.F64)
        for thr in (0.5, 0.05):
            bits = c.visibility_batch_bin(occ, src, thr)
            assert np.array_equal(vhp.unpack_bits(bits, nx), field >= thr), (nx, ny, nobs, thr)
            rc, pp, tr = c.visibility_batch_runs(occ, src, thr)
            assert np.array_equal(vhp.runs_to_bits(rc, pp, tr, nx), bits)
    c.close()


def test_row_runs_bit_exact(vhp, oracle):
    """vhp_visibility_batch_runs: the thresholded visibility as transition columns per row, equal to
    the bit form and to the oracle's fp64 field compared with >= threshold; widths that fill their
    last word, that do not, and rows wider than 1024 cells."""
    c = vhp.Context(0)
    rng = np.random.default_rng(5)
    # (rows of a multiple of four words take the 16-byte kernels: 1, 2, 4 and 8 lanes per row)
    for nx, ny, nobs, seed in ((101, 101, 10, 7), (64, 40, 6, 3), (96, 33, 0, 1), (1100, 37, 30, 2), (33, 31, 2, 1),
                               (128, 40, 5, 9), (256, 35, 6, 2), (384, 33, 8, 4), (1024, 20, 10, 6), (1000, 9, 4, 8)):
        occ = np.stack([rect_map(nx, ny, nobs, seed + k, 3, 14) for k in range(2)])
        n = 9
        smap = rng.integers(0, 2, n).astype(np.int32)
        src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        src[0] = (nx - 1, ny - 1); src[1] = (0, 0)
        ref = np.stack([oracle.compute_visibility(occ[m], sx, sy) for (sx, sy), m in zip(src, smap)])
        for thr in (0.5, 1.0, 0.0, 0.01):
            rc, pp, tr = c.visibility_batch_runs(occ, src, thr, src_map=smap)
            assert rc.shape == (n, ny) and pp.shape == (n + 1,) and pp[0] == 0 and pp[n] == len(tr) == rc.sum()
            assert (rc % 2 == 0).all()
            bits = vhp.runs_to_bits(rc, pp, tr, nx)
            assert np.array_equal(vhp.unpack_bits(bits, nx), ref >= thr), (nx, ny, thr)
            assert np.array_equal(bits, c.visibility_batch_bin(occ, src, thr, src_map=smap))
            # columns ascend strictly inside a row and end at most at nx
            k = 0
            for p in range(n):
                assert pp[p] == k
                for y in range(ny):
                    t = tr[k:k + rc[p, y]].astype(int)
                    assert (np.diff(t) > 0).all() and (len(t) == 0 or t[-1] <= nx)
                    k += rc[p, y]
    # too small a buffer: the call says how much it needs
    import ctypes as C
    occ = np.ones((1, 50, 50), np.uint8); src = np.array([[5, 5]], np.int32)
    rc = np.zeros((1, 50), np.uint16); pp = np.zeros(2, np.uint64); tr = np.zeros(10, np.uint16); used = C.c_int64(0)
    st = c.lib.vhp_visibility_batch_runs(c.h, occ.ctypes.data, 1, 50, 50, src.ctypes.data, None, 1, 0.5,
                                         rc.ctypes.data, pp.ctypes.data, tr.ctypes.data, 10, C.byref(used))
    assert st == -1 and used.value == 98   # rows 1..49: visible on [1, 50); row 0 is the never-written border
    c.close()


def test_packed_handle_expands_bit_identical(vhp):
    """vhp_visibility_batch_packed + vhp_packed_expand: the whole batch, single pairs and ranges that
    start / end inside 128-byte units (101 x 101 x 4 bytes is not a multiple of 128) rebuild exactly the
    bytes vhp_visibility_batch returns; fp32 and fp64; several chunks; a reused handle."""
    rng = np.random.default_rng(31)
    c = vhp.Context(0)
    h = None
    for nx, ny, nobs, n, dt in ((101, 101, 10, 40, vhp.F32), (1000, 1000, 15, 150, vhp.F32), (333, 77, 6, 25, vhp.F64),
                                (64, 64, 0, 9, vhp.F32), (1000, 1000, 0, 290, vhp.F64)):
        occ = np.stack([rect_map(nx, ny, nobs, 70 + k, 8, 120 if nx > 500 else 20) for k in range(2)])
        smap = rng.integers(0, 2, n).astype(np.int32)
        src = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], 1).astype(np.int32)
        want = c.visibility_batch(occ, src, src_map=smap, dtype=dt)
        h = c.visibility_batch_packed(occ, src, src_map=smap, dtype=dt, handle=h)
        assert len(h) == n and 0 < h.nbytes < want.nbytes
        got = h.expand()
        assert got.dtype == want.dtype and np.array_equal(got.view(np.uint8), want.view(np.uint8)), (nx, ny)
        for first, count in ((0, 1), (n - 1, 1), (n // 3, 5), (1, n - 2)):
            part = h.expand(first, count, threads=3 if count > 2 else 1)
            assert np.array_equal(part.view(np.uint8), want[first:first + count].view(np.uint8)), (nx, ny, first, count)
        if nx == 1000 and nobs == 0:
            assert h.nbytes < 0.1 * want.nbytes  # open maps: one element per unit and a few literal units
    with pytest.raises(vhp.VhpError):
        h.expand(0, len(h) + 1)
    h.close()
    c.close()
