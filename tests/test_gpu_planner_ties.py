"""The planner's next-source choice under exact ties on every route, against the oracle.

The cases (test_planner_ties_cpu.py, where a witness from the stepped oracle shows that each one ties, and which
kinds of tie the set covers) are maps mirrored about the source's column, row, both, or the main diagonal, sources on
the map's border, and start and end on one row or column at threshold 0.  Each runs on the three planner routes of
test_gpu_planner.py -- one persistent CTA per problem, the batch-wide first sweep, the grid route -- one problem per
call, all of one shape in one batch through prob_map, through the device entry point, and with fp32 fields; then on
the strip-partitioned planner with its strip boundaries between mirrored tied cells.  Every comparison is against
oracle.solve: light sources, path, fields, fp64 bit for bit and fp32 as the fp64 value rounded once."""
import numpy as np
import pytest

from test_gpu_giant import env, run_case  # noqa: F401  (env: the fixture run_case takes its context from)
from test_gpu_planner_dev import check, ctx, run_dev, torch, vhp  # noqa: F401  (ctx: the cta / first / grid routes)
from test_planner_ties_cpu import (GIANT_STRIPS, LINE_ITER, LINE_THR, SYM_ITER, SYM_THR, big_line_cases, giant_cases,
                                   line_cases, symmetric_cases)

pytestmark = pytest.mark.gpu
LOOP_MODES = ((1, 0), (2, 3), (3, 0))  # the graph, batches of 3 iterations, one read-back per iteration


@pytest.fixture(scope="module")
def groups(oracle):
    """[(cases, threshold, max_iter, oracle results)]: the 61 x 61 symmetric cases, the 61 x 61 line cases"""
    out = []
    for cases, thr, mi in ((symmetric_cases(), SYM_THR, SYM_ITER), (line_cases(), LINE_THR, LINE_ITER)):
        out.append((cases, thr, mi, [oracle.solve(occ, start, end, thr, mi) for _, occ, start, end in cases]))
    return out


@pytest.fixture(scope="module")
def big(oracle):
    """{name: (occ, start, end, oracle result)} of the 1000 x 1000 and 12000 x 48 line cases"""
    return {name: (occ, start, end, oracle.solve(occ, start, end, LINE_THR, LINE_ITER))
            for name, occ, start, end in big_line_cases()}


def batch_inputs(cases):
    maps = np.stack([occ for _, occ, _, _ in cases]).astype(np.uint8)
    se = np.array([start + end for _, _, start, end in cases], np.int32)
    return maps, se, np.arange(len(cases), dtype=np.int32)


def test_one_problem_per_call(ctx, vhp, groups):
    for cases, thr, mi, refs in groups:
        for (name, occ, start, end), ref in zip(cases, refs):
            try:
                check(ctx.planner_batch(occ, [start + end], threshold=thr, max_iter=mi), 0, ref)
            except AssertionError as e:
                raise AssertionError(name) from e


def test_all_cases_in_one_batch(ctx, vhp, groups):
    """One call per group, a map per problem through prob_map, fp64 and fp32 fields"""
    for cases, thr, mi, refs in groups:
        maps, se, pmap = batch_inputs(cases)
        for dtype in (vhp.F64, vhp.F32):
            r = ctx.planner_batch(maps, se, prob_map=pmap, threshold=thr, max_iter=mi, dtype=dtype)
            for k, ((name, _, _, _), ref) in enumerate(zip(cases, refs)):
                try:
                    check(r, k, ref, f32=dtype == vhp.F32)
                except AssertionError as e:
                    raise AssertionError((name, dtype)) from e


def test_device_entry_point(ctx, vhp, torch, groups):
    for cases, thr, mi, refs in groups:
        maps, se, pmap = batch_inputs(cases)
        for dtype in (vhp.F64, vhp.F32):
            r = run_dev(ctx, vhp, torch, maps, se, pmap=pmap, thr=thr, max_iter=mi, dtype=dtype)
            for k, ((name, _, _, _), ref) in enumerate(zip(cases, refs)):
                try:
                    check(r, k, ref, f32=dtype == vhp.F32)
                except AssertionError as e:
                    raise AssertionError((name, dtype)) from e


def test_line_1000(ctx, vhp, torch, big):
    """About 860 dark cells of one row tie at every iteration; the first pushed is the one nearest the source, on
    its left: not the smallest index"""
    occ, start, end, ref = big["line1000"]
    check(ctx.planner_batch(occ, [start + end], threshold=LINE_THR, max_iter=LINE_ITER), 0, ref)
    check(run_dev(ctx, vhp, torch, occ, [start + end], thr=LINE_THR, max_iter=LINE_ITER, dtype=vhp.F32), 0, ref,
          f32=True)


def test_line_12000x48_grid_route(vhp, torch, big):
    """About 11 900 cells of one row tie; the map is too wide for one CTA, so the grid route runs it by default"""
    from test_gpu_planner_dev import make_ctx
    occ, start, end, ref = big["line12000x48"]
    c = make_ctx(vhp, torch)
    check(c.planner_batch(occ, [start + end], threshold=LINE_THR, max_iter=LINE_ITER), 0, ref)
    for dtype in (vhp.F64, vhp.F32):
        r = run_dev(c, vhp, torch, occ, [start + end], thr=LINE_THR, max_iter=LINE_ITER, dtype=dtype)
        check(r, 0, ref, f32=dtype == vhp.F32)
    c.close()


@pytest.mark.parametrize("grid_sweep", [0, 2])  # single-CTA window kernel / many-CTA grid kernels
@pytest.mark.parametrize("nstrips", GIANT_STRIPS)
def test_giant_strips(env, oracle, nstrips, grid_sweep):
    """Every giant case on 1, 2, 3 and 5 strips in three loop modes.  Each case's map is mirrored about the first
    row of strip 1 of its own strip count, so there the tied cells lie in two strips"""
    from visibility_heuristic_path_planner_b200.giant import GiantPlanner
    vhp_, ctx_ = env
    for name, occ, start, end, _ in giant_cases():
        ctx_.set_grid_sweep(grid_sweep)
        gp = GiantPlanner(occ, ctx=ctx_, strips_per_rank=nstrips)
        try:
            for loop, batch in LOOP_MODES:
                try:
                    run_case(vhp_, ctx_, oracle, occ, start, end, SYM_THR, SYM_ITER, nstrips, grid_sweep, loop, batch,
                             planner=gp)
                except AssertionError as e:
                    raise AssertionError((name, loop, batch)) from e
        finally:
            gp.close()
