"""Range-limited merged visibility (vhp_visibility_merge_range_batch_dev): device time of the direct route against
the fallback and against what callers write without the call, on three workloads.  Prints one JSON line.

    python tools/merge_range_probe.py [--reps 5] [--warm 2] [--out FILE]

Paths (fp64 vmax, int32 first and count; the maps are packed once with prepare_maps_dev, as a caller with fixed
maps would):
  direct       the sweep of each source's box folds straight into the group outputs (kFmtMergeRange64), thr = 0.5
  fallback     fp64 windows of 1 GB chunks of sources (the windowed kernel) + merge_window_fold_kernel, reached
               through thr = 0.0 (no switch exists for it)
  windows      visibility_window_batch_dev into fp64 windows of every source, then a torch fold: scatter_reduce
               amax into vmax, amin into first, index_add into count, with the range and "writes" masks (thr = 0.5)
  merge        (w1000 only) visibility_merge_batch_dev of the same groups: a box of R = 1000 covers the whole map
Workloads:
  g16384   one group of 65 536 disk sensors, R = 32, on one device-generated 16384 x 16384 map (the shipped
           obstacle density, 15 rectangles of 100-200 cells per 1000^2), threshold 0.5
  c1000    256 groups x 16 disk sensors, R = 64, on one 1000 x 1000 map with the shipped obstacle settings:
           candidate sensor placements
  w1000    box, R = 1000: 64 groups x 64 sources, one shipped-settings 1000 x 1000 map per group (merge_probe's
           s64); the torch fold is left out there (the windows alone would take 131 GB)
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.  Each workload
also records whether the direct route's outputs equal the other paths' (exact).
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
from window_probe import obstacle_map  # noqa: E402


def torch_fold(torch, win, xy_t, gid_t, kid_t, outs, nx, ny, R, disk, thr):
    """the windows (n, 2R+1, 2R+1, fp64) of sources with group gid and index kid folded into outs by torch"""
    vmax, first, count = outs
    dev = win.device
    W = 2 * R + 1
    v, u = torch.meshgrid(torch.arange(W, device=dev) - R, torch.arange(W, device=dev) - R, indexing="ij")
    inr = (u * u + v * v <= R * R) if disk else torch.ones((W, W), dtype=torch.bool, device=dev)
    x = xy_t[:, 0, None, None] + u
    y = xy_t[:, 1, None, None] + v
    ok = inr & (x >= 0) & (x < nx) & (y >= 0) & (y < ny)
    cell = gid_t[:, None, None].long() * (nx * ny) + y.long() * nx + x.long()
    writes = ~(((x == 0) & (xy_t[:, 0, None, None] != 0)) | ((y == 0) & (xy_t[:, 1, None, None] != 0)))
    hit = ok & writes & (win >= thr)
    vmax.zero_()
    first.fill_(2**31 - 1)
    count.zero_()
    vmax.view(-1).scatter_reduce_(0, cell[ok], win[ok], "amax")
    k = kid_t[:, None, None].expand(-1, W, W)
    first.view(-1).scatter_reduce_(0, cell[hit], k[hit], "amin")
    first[first == 2**31 - 1] = -1
    count.view(-1).index_add_(0, cell[hit], torch.ones_like(cell[hit], dtype=torch.int32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("merge_range_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(13)
    res = dict(probe="merge_range", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731

    def shipped_maps(n):
        return torch.from_numpy(np.stack([shipped_map(g) for _ in range(n)])).to(dev)

    def workloads():
        occ_t = obstacle_map(vhp, torch, dev, 16384, 16384)
        yield "g16384", occ_t, free_sources(g, occ_t.cpu().numpy(), 65536), 65536, 32, vhp.RANGE_DISK
        occ_t = shipped_maps(1)
        yield "c1000", occ_t, free_sources(g, occ_t.cpu().numpy(), 4096), 16, 64, vhp.RANGE_DISK
        occ_t = shipped_maps(64)
        yield "w1000", occ_t, free_sources(g, occ_t.cpu().numpy(), 64), 64, 1000, vhp.RANGE_BOX

    for name, occ_t, xy, K, R, shape in workloads():
        nmaps, ny, nx = occ_t.shape
        n = xy.shape[0]
        ng = n // K
        disk = shape == vhp.RANGE_DISK
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            gm_t = torch.arange(ng, dtype=torch.int32, device=dev) if nmaps > 1 else None
            outs = [torch.empty((ng, ny, nx), dtype=torch.float64, device=dev),
                    torch.empty((ng, ny, nx), dtype=torch.int32, device=dev),
                    torch.empty((ng, ny, nx), dtype=torch.int32, device=dev)]
            ref = [torch.empty_like(o) for o in outs]
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        w = dict(groups=ng, sources_per_group=K, maps=nmaps, nx=nx, ny=ny, radius=R,
                 shape="disk" if disk else "box", threshold=0.5, paths={})

        def run(thr, o):
            return lambda: ctx.visibility_merge_range_batch_dev(occ_t, xy_t, ptr_t, thr, R, shape, vmax_t=o[0],
                                                                first_t=o[1], count_t=o[2], group_map_t=gm_t)

        w["paths"]["direct"] = T(run(0.5, outs))
        w["paths"]["fallback"] = T(run(0.0, ref))
        ctx.synchronize()
        run(0.5, outs)()
        ctx.synchronize()
        if name == "w1000":
            def merge():
                ctx.visibility_merge_batch_dev(occ_t, xy_t, ptr_t, 0.5, vmax_t=ref[0], first_t=ref[1], count_t=ref[2],
                                               group_map_t=gm_t)
            w["paths"]["merge"] = T(merge)
            ctx.synchronize()
            w["direct_equals_merge"] = bool(all(torch.equal(a, b) for a, b in zip(outs, ref)))
        else:
            W = 2 * R + 1
            smap_t = (torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
                      if nmaps > 1 else None)
            with torch.cuda.stream(stream):
                win = torch.empty((n, W, W), dtype=torch.float64, device=dev)
                gid_t = torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
                kid_t = torch.arange(n, device=dev, dtype=torch.int32) % K
            stream.synchronize()

            def windows():
                ctx.visibility_window_batch_dev(occ_t, xy_t, R, win, src_map_t=smap_t)
                torch_fold(torch, win, xy_t, gid_t, kid_t, ref, nx, ny, R, disk, 0.5)
            w["paths"]["windows"] = T(windows)
            ctx.synchronize()
            w["window_bytes"] = n * W * W * 8
            w["direct_equals_windows"] = bool(all(torch.equal(a, b) for a, b in zip(outs, ref)))
            del win
        for p in w["paths"].values():
            p["gsource_box_cells_per_s"] = n * min(2 * R + 1, nx) * min(2 * R + 1, ny) / (p["ms_median"] * 1e6)
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        del occ_t, outs, ref
        torch.cuda.empty_cache()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
