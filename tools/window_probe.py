"""Range-limited visibility (vhp_visibility_window_batch_dev): device time of the windowed route against the ways a
caller gets the same windows without it.  Prints one JSON line.

    python tools/window_probe.py [--reps 5] [--warm 2] [--out FILE]

Workloads (fp32 outputs, bit planes prepared once with vhp_prepare_maps_dev, as a caller with fixed maps would):
  w8192   16384 sources, R = 128, on one device-generated 8192 x 8192 map (1000 rectangles of 100-200 cells: the
          density of the shipped 1000 x 1000 settings).  Rows:
            window         the windowed route
            batch257       1024 maps of 257 x 257 cut from the same map, 16 sources each: the same number of cells
                           through visibility_batch_dev, i.e. the rate the one-CTA kernel reaches on maps that size
            full_and_crop  64 of the sources as whole 8192 x 8192 fields (visibility_batch_dev, 4 at a time) plus a
                           crop; reported per source (ms_per_source) next to the window row's
  c2s_R64, c2s_R500
          4096 sources on a 1000 x 1000 map with the shipped obstacle settings, against whole fields
          (visibility_batch_dev) for the same sources
  g16384  65536 sources, R = 32, on one 16384 x 16384 map (the library's largest) with the same obstacle density
Rates: window cells per second (pairs x (2R+1)^2 / time) and output bytes per second.
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.
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


def rates(r, pairs, W, esz=4):
    cells = pairs * W * W
    r["window_gcells_per_s"] = cells / (r["ms_median"] * 1e6)
    r["output_gb_per_s"] = cells * esz / (r["ms_median"] * 1e6)
    return r


def obstacle_map(vhp, torch, dev, n, seed):
    """one n x n map, (n / 1000)^2 * 15 rectangles of 100-200 cells"""
    c = vhp.Context(0)
    t = torch.empty((1, n, n), dtype=torch.uint8, device=dev)
    c.generate_environments_dev(t, int(15 * (n / 1000) ** 2), 100, 200, 100, 200, seed=seed)
    c.synchronize()
    c.close()
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("window_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(11)
    res = dict(probe="window", gpu=gpu_info(), dtype="fp32", workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731

    def window_row(occ_t, xy_t, R):
        W = 2 * R + 1
        with torch.cuda.stream(stream):
            out = torch.empty((xy_t.shape[0], W, W), dtype=torch.float32, device=dev)
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        r = rates(T(lambda: ctx.visibility_window_batch_dev(occ_t, xy_t, R, out)), xy_t.shape[0], W)
        return r, out

    # ---- 8192 x 8192, R = 128 --------------------------------------------------------------------------------
    R, n = 128, 16384
    W = 2 * R + 1
    occ_t = obstacle_map(vhp, torch, dev, 8192, 8192)
    occ = occ_t.cpu().numpy()
    xy = free_sources(g, occ, n)
    xy_t = torch.from_numpy(xy).to(dev)
    w = dict(pairs=n, radius=R, nx=8192, ny=8192, window_output_bytes=n * W * W * 4, rows={})
    r, out = window_row(occ_t, xy_t, R)
    r["ms_per_source"] = r["ms_median"] / n
    w["rows"]["window"] = r
    del out
    torch.cuda.empty_cache()
    tiles = np.stack([occ[0, (k // 32) * 255:(k // 32) * 255 + W, (k % 32) * 255:(k % 32) * 255 + W]
                      for k in range(1024)])
    t_xy = free_sources(g, tiles, 16)
    with torch.cuda.stream(stream):
        tiles_t = torch.from_numpy(np.ascontiguousarray(tiles)).to(dev)
        t_xy_t = torch.from_numpy(t_xy).to(dev)
        t_map_t = torch.arange(1024, dtype=torch.int32, device=dev).repeat_interleave(16)
        fields = torch.empty((16384, W, W), dtype=torch.float32, device=dev)
    stream.synchronize()
    ctx.prepare_maps_dev(tiles_t)
    w["rows"]["batch257"] = rates(T(lambda: ctx.visibility_batch_dev(tiles_t, t_xy_t, fields, src_map_t=t_map_t)),
                                  16384, W)
    del fields, tiles_t
    torch.cuda.empty_cache()
    ctx.prepare_maps_dev(occ_t)
    sub = xy_t[:64].contiguous()
    with torch.cuda.stream(stream):
        buf = torch.empty((4, 8192, 8192), dtype=torch.float32, device=dev)
        crops = torch.empty((64, W, W), dtype=torch.float32, device=dev)
    hs = xy[:64]
    stream.synchronize()

    def full_and_crop():
        for p0 in range(0, 64, 4):
            ctx.visibility_batch_dev(occ_t, sub[p0:p0 + 4], buf)
            pad = torch.nn.functional.pad(buf, (R, R, R, R))
            for k in range(4):
                sx, sy = int(hs[p0 + k, 0]), int(hs[p0 + k, 1])
                crops[p0 + k] = pad[k, sy:sy + W, sx:sx + W]

    r = T(full_and_crop)
    r["ms_per_source"] = r["ms_median"] / 64
    r["pairs"] = 64
    w["rows"]["full_and_crop"] = r
    del buf, crops
    torch.cuda.empty_cache()
    w["window_slowdown_vs_batch257"] = w["rows"]["window"]["ms_median"] / w["rows"]["batch257"]["ms_median"]
    res["workloads"]["w8192"] = w
    del occ_t
    torch.cuda.empty_cache()

    # ---- 1000 x 1000 shipped settings, R in {64, 500}, against whole fields ----------------------------------
    occ = shipped_map(g)[None]
    xy = free_sources(g, occ, 4096)
    with torch.cuda.stream(stream):
        occ_t = torch.from_numpy(occ).to(dev)
        xy_t = torch.from_numpy(xy).to(dev)
        fields = torch.empty((4096, 1000, 1000), dtype=torch.float32, device=dev)
    stream.synchronize()
    ctx.prepare_maps_dev(occ_t)
    full = T(lambda: ctx.visibility_batch_dev(occ_t, xy_t, fields))
    full["field_gcells_per_s"] = 4096 * 1e6 / (full["ms_median"] * 1e6)
    for R in (64, 500):
        W = 2 * R + 1
        r, out = window_row(occ_t, xy_t, R)
        res["workloads"][f"c2s_R{R}"] = dict(pairs=4096, radius=R, nx=1000, ny=1000, rows=dict(window=r, full_fields=full),
                                             window_over_full=r["ms_median"] / full["ms_median"])
        del out
        torch.cuda.empty_cache()
    del fields, occ_t
    torch.cuda.empty_cache()

    # ---- 16384 x 16384, R = 32 ----------------------------------------------------------------------------
    R, n = 32, 65536
    occ_t = obstacle_map(vhp, torch, dev, 16384, 16384)
    xy = free_sources(g, occ_t.cpu().numpy(), n)
    xy_t = torch.from_numpy(xy).to(dev)
    r, out = window_row(occ_t, xy_t, R)
    res["workloads"]["g16384"] = dict(pairs=n, radius=R, nx=16384, ny=16384, rows=dict(window=r))
    del out, occ_t
    torch.cuda.empty_cache()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
