"""Every warp-count instance of the batched tile sweep and of the persistent planner kernel against the CPU oracle.

The sweep is compiled for 1, 2, 4, 6, 8, 10 and 16 warps per CTA and the planner for 2, 4, 6 and 8.  Which one runs
depends on the map size, the batch size and the process-wide variables VHP_TILE_WARPS / VHP_PLANNER_WARPS, which the
library reads once per process.  So each forced setting runs in a worker process of its own (this file's __main__):
the test writes the inputs to an .npz, the worker makes the library calls (every whole-field sweep and planner call,
and the first call of every other output, under torch.profiler) and writes the outputs and the names of the kernels
that ran back.  The oracle and every expectation stay here.  A check of the
instance by its kernel name (sweep_tile_kernel<double, 16, 2, 0>, planner_kernel<6, 3>) keeps a misspelled or ignored
variable from passing on the default instance.  Every comparison is exact: fp64 bit for bit, fp32 the oracle's value
rounded once."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_golden, rect_map
from test_gpu_cover import check as cover_check
from test_gpu_cover import expected as cover_expected
from test_gpu_merge import check as merge_check
from test_gpu_merge import expected as merge_expected
from test_gpu_merge import make_groups
from test_gpu_merge_range import expected as merge_range_expected
from test_gpu_planner import check as planner_check
from test_window_cpu import window_of

pytestmark = pytest.mark.gpu
F32, F64, RANGE_BOX, RANGE_DISK = 0, 1, 0, 1  # the package's constants (the parent process imports it lazily)
ENV_VARS = ("VHP_TILE_WARPS", "VHP_PLANNER_WARPS", "VHP_PLANNER_FIRST", "VHP_PLANNER_ROUNDS", "VHP_SWEEP_IMPL",
            "VHP_GRID_SWEEP", "VHP_BIN_DIRECT")
TILE_WARPS = (1, 2, 4, 6, 8, 10, 16)
PLANNER_WARPS = (2, 4, 6, 8)
SWEEP_RE = re.compile(r"\bsweep_tile_kernel<(float|double), (\d+), (\d+), (\d+)>")
PLANNER_RE = re.compile(r"\bplanner_kernel<(\d+), (\d+)>")
# fp64 / fp32 sweeps of wide maps under a forced count: the instance whose CTA fits shared memory (227 KB), the
# 8-warp one otherwise.  (nx, ny = 40, dtype, forced) -> warps that run
WIDE = {(6000, F64, 10): 10, (6000, F64, 16): 8, (9000, F64, 10): 8, (9000, F64, 16): 8,
        (6000, F32, 16): 16, (9000, F32, 16): 16, (9200, F32, 10): 10, (9200, F32, 16): 8}


def other_formats_warps(w):
    """Warps of the bit, merge, window and cover sweeps under VHP_TILE_WARPS=w: those have 1-, 4- and 8-warp instances"""
    return {2: 4, 6: 4, 10: 8, 16: 8}.get(w, w)


# ---- the worker ---------------------------------------------------------------------------------------------------

def worker(d):
    """Make the library calls of d/jobs.json on the arrays of d/in.npz; write d/out.npz and d/meta.json."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import visibility_heuristic_path_planner_b200 as vhp
    from torch.profiler import ProfilerActivity, profile

    arrays = dict(np.load(os.path.join(d, "in.npz")))
    with open(os.path.join(d, "jobs.json")) as f:
        jobs = json.load(f)
    ctx = vhp.Context(0)
    ctx.set_grid_sweep(0)  # one CTA per pair whatever the batch size: the tile kernel under test
    val = lambda v: arrays[v["npz"]] if isinstance(v, dict) else v  # noqa: E731
    out, meta = {}, []
    for i, job in enumerate(jobs):
        args = [val(a) for a in job["args"]]
        kwargs = {k: val(v) for k, v in job["kwargs"].items()}
        m = dict(error=None, kernels=None)
        try:
            if job["profile"]:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    r = getattr(ctx, job["method"])(*args, **kwargs)
                    ctx.synchronize()
                m["kernels"] = sorted({e.key for e in prof.key_averages() if "Memcpy" not in e.key
                                       and "Memset" not in e.key})
            else:
                r = getattr(ctx, job["method"])(*args, **kwargs)
        except vhp.VhpError as e:
            m["error"] = f"status {e.status}: {e}"
            r = None
        if isinstance(r, dict):
            out.update({f"{i}/{k}": v for k, v in r.items()})
        elif isinstance(r, tuple):
            out.update({f"{i}/{k}": v for k, v in enumerate(r)})
        elif r is not None:
            out[f"{i}/0"] = r
        meta.append(m)
    ctx.close()
    np.savez(os.path.join(d, "out.npz"), **out)
    with open(os.path.join(d, "meta.json"), "w") as f:
        json.dump(meta, f, indent=1)


# ---- the calls a worker makes and what they must return -----------------------------------------------------------

class Batch:
    """Library calls for one worker, and per call a check of its outputs and of the kernels that ran."""

    def __init__(self):
        self.arrays, self.jobs, self.checks, self.profiled = {}, [], [], set()

    def _arg(self, v):
        if isinstance(v, np.ndarray):
            key = f"a{len(self.arrays)}"
            self.arrays[key] = v
            return {"npz": key}
        return v

    def call(self, group, method, args, kwargs, check, kernels, profile_once=None):
        """check(out): out is the dict / tuple / array the method returns; kernels(names): the profiled names.
        profile_once: a key; of the calls with the same key only the first runs under the profiler"""
        profile = profile_once is None or profile_once not in self.profiled
        self.profiled.add(profile_once)
        self.jobs.append(dict(method=method, args=[self._arg(a) for a in args],
                              kwargs={k: self._arg(v) for k, v in kwargs.items()}, profile=profile))
        self.checks.append((group, f"{method} #{len(self.jobs) - 1}", check, kernels))


def sweep_instances(names):
    """(dtype, warps, format) of every sweep_tile_kernel in the profiled names"""
    return {(m.group(1), int(m.group(2)), int(m.group(4))) for n in names for m in SWEEP_RE.finditer(n)}


def planner_instances(names):
    return {int(m.group(1)) for n in names for m in PLANNER_RE.finditer(n)}


def expect_sweep(warps, dtype=None, values=False):
    def kernels(names):
        got = sweep_instances(names)
        assert {w for _, w, _ in got} == {warps}, (warps, names)
        if dtype is not None:
            assert {t for t, _, _ in got} == {"float" if dtype == F32 else "double"}, names
        if values:
            assert {f for _, _, f in got} == {0}, names
    return kernels


def expect_planner(warps, first_sweep_warps=None):
    def kernels(names):
        assert planner_instances(names) == {warps}, (warps, names)
        got = sweep_instances(names)
        if first_sweep_warps is None:
            assert not got, names
        else:
            assert got == {("double", first_sweep_warps, 0)}, (first_sweep_warps, names)
    return kernels


def values_check(ref, dtype):
    want = ref.astype(np.float32) if dtype == F32 else ref

    def check(out):
        got = out[0]
        assert got.shape == want.shape
        bad = [(p, np.argwhere(g != w)[:3].tolist()) for p, (g, w) in enumerate(zip(got, want)) if not np.array_equal(g, w)]
        assert not bad, bad[:3]
    return check


def add_values(b, group, occ, srcs, smap, ref, warps, dtypes=(F64, F32)):
    """Whole-field sweeps of the pairs (map smap[p] or 0, source srcs[p]) against the oracle's fields ref"""
    for dt in dtypes:
        kw = dict(dtype=dt) if smap is None else dict(src_map=smap, dtype=dt)
        b.call(group, "visibility_batch", [occ, srcs], kw, values_check(ref, dt), expect_sweep(warps, dt, True))


def oracle_fields(oracle, occ, srcs, smap=None):
    occ = occ if occ.ndim == 3 else occ[None]
    smap = np.zeros(len(srcs), int) if smap is None else smap
    return np.stack([oracle.compute_visibility(occ[m], int(x), int(y)) for (x, y), m in zip(srcs, smap)])


def planner_ref(oracle, occ, se, thr, max_iter):
    return oracle.solve(np.asarray(occ, np.float64), se[:2], se[2:], thr, max_iter)


# ---- inputs and expectations, computed once ----------------------------------------------------------------------

@pytest.fixture(scope="module")
def value_cases(oracle):
    """(name, occ (nmaps, ny, nx) uint8, sources int32 (n, 2), src_map or None, oracle fields)"""
    cases = []

    def add(name, occ, srcs, smap=None):
        occ = np.asarray(occ).reshape((-1,) + np.asarray(occ).shape[-2:])
        srcs = np.asarray(srcs, np.int32).reshape(-1, 2)
        cases.append((name, (occ != 0).astype(np.uint8), srcs, smap, oracle_fields(oracle, occ, srcs, smap)))

    for nx, ny in ((1, 1), (1, 9), (9, 1), (2, 2)):
        add(f"{nx}x{ny}", np.ones((ny, nx)), [(x, y) for y in range(ny) for x in range(nx)])
    rng = np.random.default_rng(33)
    s33 = [(0, 0), (32, 32), (0, 32), (32, 0), (16, 16), (31, 5), (1, 31)]
    add("33x33", rect_map(33, 33, 4, 33, 1, 6), s33 + [tuple(rng.integers(0, 33, 2)) for _ in range(9)])
    for nx, ny in ((200, 96), (197, 70)):  # every residue of sx mod 32 (test_every_tile_alignment's sources)
        srcs = [(x, (7 * x + 3) % ny) for x in range(0, 70)] + [(nx - 1 - x, ny - 1) for x in range(0, 34)]
        add(f"align{nx}x{ny}", rect_map(nx, ny, 14, 4242 + nx, 3, 17), srcs)
    maps = np.stack([rect_map(96, 80, 10, 50 + m, 2, 12) for m in range(7)])  # test_multi_map_batch's batch
    g = np.random.default_rng(5)
    smap = g.integers(0, 7, 40).astype(np.int32)
    add("multimap", maps, np.stack([g.integers(0, 96, 40), g.integers(0, 80, 40)], axis=1), smap)
    g = np.random.default_rng(130)
    empty_srcs = [(0, 0), (129, 60), (0, 60), (129, 0), (64, 30)] + [tuple(g.integers(0, 61, 2)) for _ in range(11)]
    add("empty130x61", np.ones((61, 130)), empty_srcs)  # all lit: only the staircase and the lit fill
    dense = rect_map(150, 120, 1500, 31, 1, 3)  # 29 % of the cells blocked: dark runs everywhere
    free = np.argwhere(dense != 0)
    pick = free[np.random.default_rng(150).choice(len(free), 14, replace=False)]
    add("dense150x120", dense, [(0, 0), (149, 119)] + [(int(x), int(y)) for y, x in pick])
    shipped = oracle.generate_environment(1000, 1000, 15, 100, 200, 100, 200, 1)
    add("shipped1000", shipped, [(0, 0), (999, 999), (0, 999), (999, 0), (50, 50), (0, 500), (500, 0)])
    big = oracle.generate_environment(2100, 1300, 60, 20, 160, 20, 160, 5)
    add("2100x1300", big, [(0, 0), (2099, 1299), (0, 1299), (2099, 0), (1050, 650), (0, 700), (900, 0)])
    return cases


@pytest.fixture(scope="module")
def format_case(oracle):
    """One set of maps and groups for the bit, row-run, merge, window and cover outputs"""
    nx, ny = 101, 77
    rng = np.random.default_rng(101)
    occ = np.stack([rect_map(nx, ny, 10, 90 + m, 3, 14) for m in range(3)]).astype(np.uint8)
    sizes = [0, 1, 2, 7, 33, 0, 2]  # empty groups, one source, duplicates (make_groups)
    srcs, ptr = make_groups(rng, nx, ny, occ[1], sizes)
    gmap = np.array([g % 3 for g in range(len(sizes))], np.int32)
    pmap = np.repeat(gmap, np.diff(ptr)).astype(np.int32)
    return dict(nx=nx, ny=ny, occ=occ, srcs=srcs, ptr=ptr, gmap=gmap, pmap=pmap,
                fields=oracle_fields(oracle, occ, srcs, pmap))


@pytest.fixture(scope="module")
def planner_cases(oracle):
    """(occ, start_end, prob_map or None, threshold, max_iter, oracle results): the planner.npz goldens, the random
    problems of test_random_problems_vs_oracle"""
    cases = []
    g = load_golden("planner.npz")
    maps = np.stack([oracle.generate_environment(101, 101, 10, 10, 20, 10, 20, s) for s in range(1, 7)])
    se = np.tile(np.array([5, 5, 95, 95], np.int32), (6, 1))
    refs = [dict(status=int(g[f"s101_{s}_status"][0]), nb_of_sources=int(g[f"s101_{s}_status"][1]),
                 light_sources=g[f"s101_{s}_ls"], path=g[f"s101_{s}_path"], path_length=g[f"s101_{s}_len"][0],
                 vg=g[f"s101_{s}_vg"], came=g[f"s101_{s}_came"], vis=g[f"s101_{s}_vis"]) for s in range(1, 7)]
    cases.append((maps, se, np.arange(6, dtype=np.int32), 0.25, 100, refs))
    rng = np.random.default_rng(77)
    for trial in range(6):
        nx, ny = int(rng.integers(20, 200)), int(rng.integers(20, 200))
        occ = rect_map(nx, ny, int(rng.integers(0, 30)), 500 + trial, 2, 14)
        se = np.stack([rng.integers(0, nx, 8), rng.integers(0, ny, 8), rng.integers(0, nx, 8),
                       rng.integers(0, ny, 8)], axis=1).astype(np.int32)
        thr = float(rng.choice([0.0, 0.2, 0.5, 0.9, 1.0]))
        cases.append((occ, se, None, thr, 12, [planner_ref(oracle, occ, s, thr, 12) for s in se]))
    return cases


@pytest.fixture(scope="module")
def maze_case(oracle):
    """maze_5 at max_iter 150: the planner stalls on one cell and takes the fixed-point fast-forward"""
    g = load_golden("maze5.npz")
    ny, nx = g["shape"]
    occ = np.unpackbits(g["occ_bits"])[: ny * nx].reshape(ny, nx)
    se = np.array([tuple(g["start"]) + tuple(g["end"])], np.int32)
    ref = planner_ref(oracle, occ, se[0], 0.25, 150)
    assert ref["status"] == 5 and ref["nb_of_sources"] == 151
    return occ, se, None, 0.25, 150, [ref]


@pytest.fixture(scope="module")
def wide_cases(oracle):
    """Maps of 6000, 9000 and 9200 x 40: sources and planner problems, with the oracle's results"""
    cases = {}
    for nx in (6000, 9000, 9200):
        occ = rect_map(nx, 40, nx // 40, nx, 4, 30)
        free = np.argwhere(occ != 0)
        pick = free[np.random.default_rng(nx).choice(len(free), 8, replace=False)]
        occ[0, 0] = occ[39, nx - 1] = occ[20, nx // 2] = 1
        srcs = np.array([(0, 0), (nx - 1, 39), (nx // 2, 20)] + [(int(x), int(y)) for y, x in pick[:3]], np.int32)
        se = np.array([(0, 0, nx - 1, 39), (nx // 2, 20, 0, 0)] + [(int(pick[k][1]), int(pick[k][0]), int(pick[k + 4][1]),
                                                                    int(pick[k + 4][0])) for k in range(2)], np.int32)
        cases[nx] = (occ.astype(np.uint8), srcs, oracle_fields(oracle, occ, srcs),
                     se, [planner_ref(oracle, occ, s, 0.3, 12) for s in se])
    return cases


@pytest.fixture(scope="module")
def vhp():
    import visibility_heuristic_path_planner_b200 as m
    return m


def add_planner(b, group, case, kernels):
    occ, se, pmap, thr, max_iter, refs = case

    def check(r):
        for k, ref in enumerate(refs):
            planner_check(r, k, ref)
    kw = dict(threshold=thr, max_iter=max_iter) if pmap is None else dict(prob_map=pmap, threshold=thr,
                                                                          max_iter=max_iter)
    b.call(group, "planner_batch", [np.asarray(occ, np.uint8), se], kw, check, kernels)


def add_formats(b, vhp, fc, w):
    """Bits, row runs, windows, merge, range-limited merge (box and disk) and greedy cover under VHP_TILE_WARPS=w"""
    nx, ny, occ, srcs, ptr, gmap, pmap, fields = (fc[k] for k in ("nx", "ny", "occ", "srcs", "ptr", "gmap", "pmap",
                                                                    "fields"))
    nw = other_formats_warps(w)
    for thr in (0.5, 1.0, 1e-9):
        def bits_check(out, thr=thr):
            assert np.array_equal(vhp.unpack_bits(out[0], nx), fields >= thr), thr
            assert not np.unpackbits(out[0].view(np.uint8), axis=-1, bitorder="little")[..., nx:].any()

        def runs_check(out, thr=thr):
            rc, pp, tr = out[0], out[1], out[2]
            assert pp[0] == 0 and pp[-1] == len(tr) == rc.sum() and (rc % 2 == 0).all()
            assert np.array_equal(vhp.unpack_bits(vhp.runs_to_bits(rc, pp, tr, nx), nx), fields >= thr), thr
        b.call("formats", "visibility_batch_bin", [occ, srcs, thr], dict(src_map=pmap), bits_check,
               expect_sweep(nw, F32), "bin")
        b.call("formats", "visibility_batch_runs", [occ, srcs, thr], dict(src_map=pmap), runs_check,
               expect_sweep(nw, F32), "runs")
        for dt in (F64, F32):
            want = merge_expected(fields, srcs, ptr, thr, (ny, nx))
            b.call("formats", "visibility_merge_batch", [occ, srcs, ptr, thr], dict(group_map=gmap, dtype=dt),
                   lambda r, want=want, dt=dt, thr=thr: merge_check(r, want, dt == F32, ("merge", thr, dt)),
                   expect_sweep(nw, F64), ("merge", dt))
    for i, R in enumerate((0, 16, 31, 33)):
        dt = (F64, F32)[i % 2]
        want_w = np.stack([window_of(f, int(x), int(y), R) for f, (x, y) in zip(fields, srcs)])
        b.call("formats", "visibility_window_batch", [occ, srcs, R], dict(src_map=pmap, dtype=dt),
               values_check(want_w, dt), expect_sweep(nw, dt), ("window", dt))
        for disk in (False, True):
            shape = RANGE_DISK if disk else RANGE_BOX
            for thr in (0.5, 1.0, 1e-9):
                want = merge_range_expected(fields, srcs, ptr, thr, (ny, nx), R, disk)
                b.call("formats", "visibility_merge_range_batch", [occ, srcs, ptr, thr, R, shape],
                       dict(group_map=gmap, dtype=dt),
                       lambda r, want=want, dt=dt, what=(R, disk, thr, dt): merge_check(r, want, dt == F32, what),
                       expect_sweep(nw, F64), ("merge_range", dt))
                cw = cover_expected(fields, srcs, ptr, thr, R, disk, 5)
                b.call("formats", "visibility_cover_greedy_batch", [occ, srcs, ptr, 5, thr, R, shape],
                       dict(group_map=gmap), lambda r, cw=cw, what=(R, disk, thr): cover_check(vhp, r, cw, nx, what),
                       expect_sweep(nw, F32), "cover")


# ---- running a worker ---------------------------------------------------------------------------------------------

class Results:
    def __init__(self, batch, out, meta):
        self.batch, self.out, self.meta = batch, out, meta

    def verify(self, group):
        n = 0
        for i, (g, name, check, kernels) in enumerate(self.batch.checks):
            if g != group:
                continue
            assert self.meta[i]["error"] is None, (name, self.meta[i]["error"])
            keys = sorted((k for k in self.out if k.startswith(f"{i}/")), key=lambda k: k.split("/")[1])
            r = {k.split("/")[1]: self.out[k] for k in keys}
            if set(r) <= {"0", "1", "2"}:
                r = [r[str(j)] for j in range(len(r))]
            check(r)
            if self.meta[i]["kernels"] is not None:
                kernels(self.meta[i]["kernels"])
            n += 1
        assert n > 0, group


@pytest.fixture(scope="module")
def run_worker(tmp_path_factory):
    """run_worker(name, env, batch) -> Results; one worker process per name, run on first use"""
    done = {}

    def run(name, env_set, batch):
        if name in done:
            return done[name]
        d = tmp_path_factory.mktemp(name)
        np.savez(d / "in.npz", **batch.arrays)
        with open(d / "jobs.json", "w") as f:
            json.dump(batch.jobs, f)
        env = {k: v for k, v in os.environ.items() if k not in ENV_VARS}
        env.update(env_set)
        cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--worker",
                                                                               str(d)]
        p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, (name, p.returncode, p.stderr[-3000:])
        with np.load(d / "out.npz") as z:
            out = {k: z[k] for k in z.files}
        os.remove(d / "out.npz")  # large; meta.json keeps the kernel names
        os.remove(d / "in.npz")
        with open(d / "meta.json") as f:
            meta = json.load(f)
        done[name] = Results(batch, out, meta)
        return done[name]
    return run


@pytest.fixture(scope="module")
def tile_run(run_worker, vhp, value_cases, format_case, planner_cases, wide_cases):
    """Worker under VHP_TILE_WARPS=w (and VHP_PLANNER_FIRST=2: the planner's first sweep is a batch-wide tile sweep)"""
    def run(w):
        b = Batch()
        for name, occ, srcs, smap, ref in value_cases:
            add_values(b, "values", occ, srcs, smap, ref, w)
        add_formats(b, vhp, format_case, w)
        for case in planner_cases:
            add_planner(b, "planner_first", case, expect_planner(8, w))
        if w in (10, 16):  # last: where a CTA of w warps would not fit, the parent commit failed these calls
            for nx, (occ, srcs, ref, se, prefs) in wide_cases.items():
                for dt in (F64, F32):
                    if (nx, dt, w) in WIDE:
                        add_values(b, "wide", occ, srcs, None, ref, WIDE[(nx, dt, w)], (dt,))
                if (nx, F64, w) in WIDE:
                    add_planner(b, "wide", (occ, se, None, 0.3, 12, prefs), expect_planner(8, WIDE[(nx, F64, w)]))
        return run_worker(f"tile{w}", {"VHP_TILE_WARPS": str(w), "VHP_PLANNER_FIRST": "2"}, b)
    return run


# ---- the tests ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("w", TILE_WARPS)
def test_values_sweep(tile_run, w):
    """fp64 and fp32 fields of tiny maps, every tile alignment, a multi-map batch, an empty and a dense map, the
    shipped 1000^2 environment and a 2100 x 1300 map, on the w-warp instance"""
    tile_run(w).verify("values")


@pytest.mark.parametrize("w", TILE_WARPS)
def test_bits_runs_merge_windows_cover(tile_run, w):
    """The other outputs of the tile sweep under a forced count: 2 and 6 run their 4-warp instance, 10 and 16 their
    8-warp one"""
    tile_run(w).verify("formats")


@pytest.mark.parametrize("w", TILE_WARPS)
def test_planner_first_sweep(tile_run, w):
    """VHP_PLANNER_FIRST=2: every problem's first sweep is a batch-wide tile sweep on the w-warp instance"""
    tile_run(w).verify("planner_first")


@pytest.mark.parametrize("w", [10, 16])
def test_forced_count_beyond_shared_memory(tile_run, w):
    """fp64 sweeps (and the planner's first sweep) of 6000 and 9000 x 40 maps and fp32 ones of 9200 x 40 under a
    count whose CTA does not fit 227 KB of shared memory run the 8-warp instance instead of failing; where it fits,
    the forced instance runs"""
    tile_run(w).verify("wide")


@pytest.mark.parametrize("w", PLANNER_WARPS)
def test_planner_warps(run_worker, planner_cases, maze_case, w):
    b = Batch()
    for case in planner_cases + [maze_case]:
        add_planner(b, "planner", case, expect_planner(w))
    run_worker(f"planner{w}", {"VHP_PLANNER_WARPS": str(w)}, b).verify("planner")


def pool_of_pairs(oracle, nx, ny, nmaps, per_map, seed):
    """nmaps maps and per_map distinct sources on each, with their oracle fields: batches draw from these pairs"""
    occ = np.stack([rect_map(nx, ny, max(1, nx * ny // 300), seed + m, 2, 9) for m in range(nmaps)]).astype(np.uint8)
    rng = np.random.default_rng(seed)
    smap, srcs = [], []
    for m in range(nmaps):
        cells = rng.choice(nx * ny, per_map, replace=False)
        cells[:2] = (0, nx * ny - 1)
        smap += [m] * per_map
        srcs += [(int(c % nx), int(c // nx)) for c in cells]
    smap, srcs = np.array(smap, np.int32), np.array(srcs, np.int32)
    return occ, srcs, smap, oracle_fields(oracle, occ, srcs, smap)


def draw(pool, n, seed):
    occ, srcs, smap, ref = pool
    idx = np.random.default_rng(seed).permutation(np.resize(np.arange(len(srcs)), n))
    return occ, srcs[idx], smap[idx], ref[idx]


def test_ignored_values_run_the_automatic_instances(run_worker, oracle, planner_cases):
    """VHP_TILE_WARPS=3 and VHP_PLANNER_WARPS=5 are not instances: the automatic choices run (8, 4 and 1 warps by
    batch size, 8-warp planner)"""
    b = Batch()
    pool = pool_of_pairs(oracle, 64, 50, 4, 75, 640)
    for n, warps in ((40, 8), (400, 4), (2400, 1)):
        occ, srcs, smap, ref = draw(pool, n, n)
        add_values(b, "values", occ, srcs, smap, ref, warps)
    add_planner(b, "values", planner_cases[0], expect_planner(8))
    run_worker("ignored", {"VHP_TILE_WARPS": "3", "VHP_PLANNER_WARPS": "5"}, b).verify("values")


@pytest.mark.parametrize("nx, ny, n, warps", [(64, 50, 296, 8), (64, 50, 297, 4), (64, 50, 2367, 4), (64, 50, 2368, 1),
                                              (512, 24, 2368, 1), (513, 24, 2368, 8)])
def test_automatic_choice_at_its_boundaries(vhp, oracle, nx, ny, n, warps):
    """In this process, with no variable set: the batch size and map size where the automatic warp count changes,
    each side against the oracle and identified by the kernel's name"""
    from torch.profiler import ProfilerActivity, profile
    if os.environ.get("VHP_TILE_WARPS"):
        pytest.skip("VHP_TILE_WARPS is set for this process")
    occ, srcs, smap, ref = draw(pool_of_pairs(oracle, nx, ny, 3, 100, nx + ny), n, n)
    c = vhp.Context(0)
    for dt in (F64, F32):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = c.visibility_batch(occ, srcs, src_map=smap, dtype=dt)
            c.synchronize()
        values_check(ref, dt)([out])
        expect_sweep(warps, dt, True)([e.key for e in prof.key_averages()])
    c.close()


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--worker":
        worker(sys.argv[2])
    else:
        sys.exit(f"usage: {sys.argv[0]} --worker DIR")
