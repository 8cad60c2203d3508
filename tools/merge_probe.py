"""Merged visibility of source groups (vhp_visibility_merge_batch_dev): device time of three ways to get vmax /
first / count per group, on three workloads.  Prints one JSON line.

    python tools/merge_probe.py [--reps 5] [--warm 2] [--out FILE]

Paths:
  direct    the sweeps fold straight into the group outputs (kFmtMerge*, relaxed red atomics), thr = 0.5
  fallback  chunks of fp64 fields (ctx->b_bin) + merge_fold_kernel; reached through thr = 0.0 (the same sweeps and
            the same fold loop as any threshold: no switch exists for it)
  fields    what a caller writes without the merge call: visibility_batch_dev (fp64) into K fields per group,
            then torch max / first / count reductions, chunked to 4 GB of fields
Workloads:
  c4     2048 device-generated 256 x 256 maps (12 rectangles of 8-40 cells) x 16 sources, one group per map
  s64    64 groups x 64 sources, one 1000 x 1000 map per group with the shipped obstacle settings (15 rectangles
         of 100-200 cells)
  one4k  one group of 4096 sources on an empty 1000 x 1000 map (every sweep folds into the same 8 MB field)
Two more rows show what bounds the direct route: sweep_bits_only (the same sweeps writing one bit per cell, the
sweep's own cost) and direct_vmax_only (one atomic per lit cell instead of three).
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=plim, sm_max_clock=clk)
    except Exception as e:  # noqa: BLE001
        return dict(error=str(e))


def shipped_map(g, n=1000):
    m = np.ones((n, n), np.uint8)
    for _ in range(15):
        x, y = int(g.integers(1, n)), int(g.integers(1, n))
        w, h = int(g.integers(100, 201)), int(g.integers(100, 201))
        m[y:y + h, x:x + w] = 0
    return m


def free_sources(g, occ, per):
    """per free-cell sources on each map of occ (nmaps, ny, nx) -> int32 (nmaps * per, 2)."""
    nmaps, ny, nx = occ.shape
    out = np.zeros((nmaps * per, 2), np.int32)
    flat = occ.reshape(nmaps, -1) != 0
    for m in range(nmaps):
        free = np.flatnonzero(flat[m])
        pick = free[g.integers(0, len(free), per)]
        out[m * per:(m + 1) * per, 0] = pick % nx
        out[m * per:(m + 1) * per, 1] = pick // nx
    return out


def workloads(vhp, torch, dev):
    g = np.random.default_rng(7)
    c = vhp.Context(0)
    t = torch.empty((2048, 256, 256), dtype=torch.uint8, device=dev)
    c.generate_environments_dev(t, 12, 8, 40, 8, 40, seed=4321)
    c.synchronize()
    c.close()
    occ = t.cpu().numpy()
    yield "c4", occ, free_sources(g, occ, 16), 16
    occ = np.stack([shipped_map(g) for _ in range(64)])
    yield "s64", occ, free_sources(g, occ, 64), 64
    occ = np.ones((1, 1000, 1000), np.uint8)
    yield "one4k", occ, free_sources(g, occ, 4096), 4096


def fields_path(torch, c, occ_t, xy_t, K, thr, outs, buf):
    """visibility_batch_dev into fp64 fields, then the torch reductions; groups of K consecutive sources, group g
    on map g (or map 0 when there is one map)."""
    nmaps, ny, nx = occ_t.shape
    n = xy_t.shape[0]
    C = buf.shape[0]
    vmax, first, count = outs
    for s0 in range(0, n, C):
        s1 = min(n, s0 + C)
        f = buf[: s1 - s0]
        smap = None
        if nmaps > 1:
            smap = torch.div(torch.arange(s0, s1, device=xy_t.device, dtype=torch.int32), K, rounding_mode="floor")
        c.visibility_batch_dev(occ_t, xy_t[s0:s1], f, src_map_t=smap)
        hit = f >= thr
        hit[xy_t[s0:s1, 0] != 0, :, 0] = False  # the never-written border of each sweep
        hit[xy_t[s0:s1, 1] != 0, 0, :] = False
        if K <= C:  # whole groups in the chunk
            g0, ng = s0 // K, (s1 - s0) // K
            fv = f.view(ng, K, ny, nx)
            hv = hit.view(ng, K, ny, nx)
            vmax[g0:g0 + ng] = fv.max(1).values
            count[g0:g0 + ng] = hv.sum(1, dtype=torch.int32)
            first[g0:g0 + ng] = torch.where(hv.any(1), torch.argmax(hv.to(torch.uint8), 1).to(torch.int32), -1)
        else:  # one group over several chunks
            g = s0 // K
            k0 = s0 - g * K
            if k0 == 0:
                vmax[g].zero_()
                first[g].fill_(-1)
                count[g].zero_()
            torch.maximum(vmax[g], f.max(0).values, out=vmax[g])
            count[g] += hit.sum(0, dtype=torch.int32)
            new = (first[g] < 0) & hit.any(0)
            first[g][new] = (k0 + torch.argmax(hit.to(torch.uint8), 0).to(torch.int32))[new]


def timed(torch, stream, fn, reps, warm):
    ts = []
    with torch.cuda.stream(stream):  # the library and the torch reductions on one stream
        for _ in range(warm):
            fn()
        stream.synchronize()
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            ts.append(a.elapsed_time(b))
    return dict(ms_median=float(np.median(ts)), ms_min=float(min(ts)), ms_max=float(max(ts)), reps=reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("merge_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    res = dict(probe="merge", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    for name, occ, xy, K in workloads(vhp, torch, dev):
        nmaps, ny, nx = occ.shape
        n = xy.shape[0]
        ng = n // K
        cells = ny * nx
        with torch.cuda.stream(stream):
            occ_t = torch.from_numpy(occ).to(dev)
            xy_t = torch.from_numpy(xy).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            gm_t = torch.arange(ng, dtype=torch.int32, device=dev) if nmaps > 1 else None
            outs = [torch.empty((ng, ny, nx), dtype=torch.float64, device=dev),
                    torch.empty((ng, ny, nx), dtype=torch.int32, device=dev),
                    torch.empty((ng, ny, nx), dtype=torch.int32, device=dev)]
            ref = [torch.empty_like(o) for o in outs]
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)  # the bit planes once, as a caller with fixed maps would
        w = dict(groups=ng, sources_per_group=K, maps=nmaps, nx=nx, ny=ny, source_cells=n * cells,
                 merged_output_bytes=ng * cells * 16, paths={})

        def merge(thr):
            return lambda: ctx.visibility_merge_batch_dev(occ_t, xy_t, ptr_t, thr, vmax_t=outs[0], first_t=outs[1],
                                                          count_t=outs[2], group_map_t=gm_t)

        for path, thr in (("direct", 0.5), ("fallback", 0.0)):
            r = timed(torch, stream, merge(thr), args.reps, args.warm)
            r["thr"] = thr
            r["gsource_cells_per_s"] = n * cells / (r["ms_median"] * 1e6)
            r["output_bytes"] = ng * cells * 16
            w["paths"][path] = r
        # what bounds the direct route: the same sweeps storing one bit per cell (almost no stores: the sweep's own
        # cost) and the direct route with vmax alone (one atomic per lit cell instead of three)
        with torch.cuda.stream(stream):
            bits_t = torch.empty((n, ny, (nx + 31) // 32), dtype=torch.int32, device=dev)
        smap_t = (torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
                  if nmaps > 1 else None)
        r = timed(torch, stream, lambda: ctx.visibility_batch_bin_dev(occ_t, xy_t, 0.5, bits_t, src_map_t=smap_t),
                  args.reps, args.warm)
        r["gsource_cells_per_s"] = n * cells / (r["ms_median"] * 1e6)
        w["paths"]["sweep_bits_only"] = r
        r = timed(torch, stream, lambda: ctx.visibility_merge_batch_dev(occ_t, xy_t, ptr_t, 0.5, vmax_t=outs[0],
                                                                        group_map_t=gm_t), args.reps, args.warm)
        r["gsource_cells_per_s"] = n * cells / (r["ms_median"] * 1e6)
        w["paths"]["direct_vmax_only"] = r
        del bits_t
        ctx.synchronize()
        # the fields path, checked against the direct route at the same threshold
        chunk = max(1, min(n, (4 << 30) // (cells * 8)))
        if K <= chunk:
            chunk = (chunk // K) * K
        with torch.cuda.stream(stream):
            buf = torch.empty((chunk, ny, nx), dtype=torch.float64, device=dev)
        stream.synchronize()
        r = timed(torch, stream, lambda: fields_path(torch, ctx, occ_t, xy_t, K, 0.5, ref, buf), args.reps, args.warm)
        r["thr"] = 0.5
        r["gsource_cells_per_s"] = n * cells / (r["ms_median"] * 1e6)
        r["output_bytes"] = n * cells * 8 + ng * cells * 16  # K fields per group, then the merged outputs
        w["paths"]["fields"] = r
        ctx.prepare_maps_dev(occ_t)
        merge(0.5)()
        ctx.synchronize()
        w["direct_equals_fields"] = bool(all(torch.equal(a, b) for a, b in zip(outs, ref)))
        res["workloads"][name] = w
        del buf, occ_t, outs, ref
        torch.cuda.empty_cache()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
