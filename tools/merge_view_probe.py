"""Directional merged visibility (vhp_visibility_merge_view_batch_dev): device time of the direct route against the
range merge on the same positions, the fallback, and what callers write without the call, on three workloads.
Prints one JSON line per workload, and the whole result at the end.

    python tools/merge_view_probe.py [--reps 5] [--warm 2] [--out FILE]

Paths (fp64 vmax, int32 first and count; the maps are packed once with prepare_maps_dev):
  direct     the sweep of each source's box folds its cells in view straight into the group outputs
             (kFmtMergeView64), thr = 0.5
  range      vhp_visibility_merge_range_batch_dev of the same positions (omnidirectional), thr = 0.5
  fallback   fp64 windows of 1 GB chunks of sources + merge_window_fold_kernel<false, true>, reached through
             thr = 0.0 (no switch exists for it)
  windows    visibility_window_batch_dev into fp64 windows of every source, multiplied by the view mask in torch,
             then merge_range_probe's torch fold (scatter_reduce amax / amin, index_add), thr = 0.5
Workloads:
  omni       merge_range_probe's g16384 (65 536 free positions, one group, R = 32 disk) with every view a == b, r = R:
             the cost of the view test against the range merge on identical work
  cam16384m  one group of 8192 free positions x 8 headings of 90 degrees (65 536 sources), R = 32 disk, on the same
             device-generated 16384 x 16384 map, threshold 0.5
  cam1000m   256 groups x (4 positions x 4 headings of 90 degrees), R = 64 disk, one shipped-settings 1000 x 1000 map
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.  Each workload
records whether the direct route's outputs equal the torch path's (and on omni, the range merge's on both routes),
exactly.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from merge_probe import free_sources, gpu_info, shipped_map, timed  # noqa: E402
from merge_range_probe import torch_fold  # noqa: E402
from window_probe import obstacle_map  # noqa: E402


def torch_view_mask(torch, views_t, R, disk):
    """(n, 2R+1, 2R+1) bool: the window cells in each source's view (the rule of vhp_visibility_merge_view_batch)"""
    dev = views_t.device
    W = 2 * R + 1
    v, u = torch.meshgrid(torch.arange(W, device=dev) - R, torch.arange(W, device=dev) - R, indexing="ij")
    r, ax, ay, bx, by = (views_t[:, i, None, None].long() for i in range(5))
    rng = (u * u + v * v <= r * r) if disk else (torch.maximum(u.abs(), v.abs()) <= r)
    c1 = ax * v - ay * u >= 0
    c2 = u * by - v * bx >= 0
    both = (ax * by - ay * bx) > 0
    return rng & torch.where(both, c1 & c2, c1 | c2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("merge_view_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(13)
    res = dict(probe="merge_view", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731

    def cameras(pos, headings, R):
        xy = np.repeat(pos, len(headings), 0).astype(np.int32)
        views = vhp.sensor_views(np.tile(np.asarray(headings, np.float64), len(pos)), 90, R)
        return xy, views

    def workloads():
        occ_t = obstacle_map(vhp, torch, dev, 16384, 16384)
        occ = occ_t.cpu().numpy()
        xy = free_sources(g, occ, 65536)  # (first, so that the positions are merge_range_probe's g16384)
        yield "omni", occ_t, xy, np.tile(np.array([[32, 1, 0, 1, 0]], np.int32), (len(xy), 1)), 65536, 32
        xy, views = cameras(free_sources(g, occ, 8192), [45.0 * j for j in range(8)], 32)
        yield "cam16384m", occ_t, xy, views, 65536, 32
        del occ_t
        occ_t = torch.from_numpy(shipped_map(g)[None]).to(dev)
        xy, views = cameras(free_sources(g, occ_t.cpu().numpy(), 1024), [0.0, 90.0, 180.0, 270.0], 64)
        yield "cam1000m", occ_t, xy, views, 16, 64

    shape = vhp.RANGE_DISK
    for name, occ_t, xy, views, K, R in workloads():
        nmaps, ny, nx = occ_t.shape
        n = xy.shape[0]
        ng = n // K
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            views_t = torch.from_numpy(views).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            mk = lambda: [torch.empty((ng, ny, nx), dtype=torch.float64, device=dev),  # noqa: E731
                          torch.empty((ng, ny, nx), dtype=torch.int32, device=dev),
                          torch.empty((ng, ny, nx), dtype=torch.int32, device=dev)]
            outs, ref = mk(), mk()
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        w = dict(groups=ng, sources_per_group=K, maps=nmaps, nx=nx, ny=ny, radius=R, shape="disk", threshold=0.5,
                 paths={})

        def view(thr, o):
            return lambda: ctx.visibility_merge_view_batch_dev(occ_t, xy_t, views_t, ptr_t, thr, R, shape, vmax_t=o[0],
                                                               first_t=o[1], count_t=o[2])

        def rng(thr, o):
            return lambda: ctx.visibility_merge_range_batch_dev(occ_t, xy_t, ptr_t, thr, R, shape, vmax_t=o[0],
                                                                first_t=o[1], count_t=o[2])

        w["paths"]["direct"] = T(view(0.5, outs))
        w["paths"]["range"] = T(rng(0.5, ref))
        ctx.synchronize()
        if name == "omni":
            w["direct_equals_range"] = bool(all(torch.equal(a, b) for a, b in zip(outs, ref)))
        w["paths"]["fallback"] = T(view(0.0, ref))
        ctx.synchronize()
        if name == "omni":
            rng(0.0, outs)()
            ctx.synchronize()
            w["fallback_equals_range_fallback"] = bool(all(torch.equal(a, b) for a, b in zip(outs, ref)))
        view(0.5, outs)()
        ctx.synchronize()
        W = 2 * R + 1
        with torch.cuda.stream(stream):
            win = torch.empty((n, W, W), dtype=torch.float64, device=dev)
            gid_t = torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
            kid_t = torch.arange(n, device=dev, dtype=torch.int32) % K
        stream.synchronize()

        def windows():
            ctx.visibility_window_batch_dev(occ_t, xy_t, R, win)
            win.mul_(torch_view_mask(torch, views_t, R, True))
            torch_fold(torch, win, xy_t, gid_t, kid_t, ref, nx, ny, R, True, 0.5)
        w["paths"]["windows"] = T(windows)
        ctx.synchronize()
        w["window_bytes"] = n * W * W * 8
        w["direct_equals_windows"] = bool(all(torch.equal(a, b) for a, b in zip(outs, ref)))
        del win
        for p in w["paths"].values():
            p["gsource_box_cells_per_s"] = n * min(W, nx) * min(W, ny) / (p["ms_median"] * 1e6)
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        del outs, ref
        torch.cuda.empty_cache()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
