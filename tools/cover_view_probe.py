"""Directional greedy sensor placement (vhp_visibility_cover_greedy_view_batch_dev): device time of camera placement
workloads and of the mask pass on its own.  Prints one JSON line.

    python tools/cover_view_probe.py [--reps 5] [--warm 2] [--out FILE]

Workloads (maps packed once with prepare_maps_dev; threshold 0.5; random uint8 weights, a fifth of them 0):
  cam16384  8192 free positions x 8 headings (0, 45, .., 315 degrees) of a 90 degree view = 65 536 candidates in one
            problem, R = 32 disk, on cover_probe.py's 16384^2 map, k = 256, m = 1 and 2
  cam1000   256 problems x (16 positions x 4 headings of 90 degrees), R = 64 disk, on the shipped-settings 1000^2 map,
            k = 8, m = 1 and 2
  omni      cover_mfold_probe.py's g16384 (65 536 free candidates, R = 32 disk, k = 256, m = 2) with omnidirectional
            views (a == b, r = R) against vhp_visibility_cover_greedy_mfold_batch_dev: the two must be equal, and the
            difference is what the view pass costs
On the camera workloads the call runs against a torch greedy over view-masked fp64 windows (visibility_window_batch_dev)
that recomputes every gain each round; pick, gain, npicked and count must be exactly equal.  `kernels` is the device
time of one call per kernel (torch.profiler, a run of its own).  Times are CUDA events on the context's stream after
warm-up: median, min and max over the repeats.
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

from cover_mfold_probe import kernel_times  # noqa: E402
from cover_weighted_probe import IDX, record_picks  # noqa: E402
from merge_probe import free_sources, gpu_info, shipped_map, timed  # noqa: E402
from window_probe import obstacle_map  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("cover_view_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(17)
    res = dict(probe="cover_view", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731
    thr = 0.5
    occ16 = obstacle_map(vhp, torch, dev, 16384, 16384)
    occ1 = torch.from_numpy(shipped_map(g)[None]).to(dev)

    def cameras(occ_t, nprob, npos, nhead, R):
        """candidates: per problem npos free positions x nhead headings of a 90 degree view, position-major"""
        xy = np.repeat(free_sources(g, occ_t.cpu().numpy(), nprob * npos), nhead, axis=0)
        heads = np.tile(np.arange(nhead) * (360.0 / nhead), nprob * npos)
        return xy, vhp.sensor_views(heads, 90, R)

    def weights(nprob, ny, nx):
        wrng = np.random.default_rng(29)
        wr = wrng.integers(0, 256, (nprob, ny, nx), dtype=np.uint8)
        wr[wrng.random((nprob, ny, nx)) < 0.2] = 0
        return torch.from_numpy(wr).to(dev)

    for name, occ_t, nprob, npos, nhead, R, k in (("cam16384", occ16, 1, 8192, 8, 32, 256),
                                                  ("cam1000", occ1, 256, 16, 4, 64, 8)):
        _, ny, nx = occ_t.shape
        xy, views = cameras(occ_t, nprob, npos, nhead, R)
        n = xy.shape[0]
        K = n // nprob
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            v_t = torch.from_numpy(views).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            gid = torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
            kid = torch.arange(n, device=dev, dtype=torch.int32) % K
            w_rand = weights(nprob, ny, nx)
            o = [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                 torch.empty((nprob, k), dtype=torch.int64, device=dev),
                 torch.empty((nprob,), dtype=torch.int32, device=dev),
                 torch.empty((nprob, ny, nx), dtype=torch.uint8, device=dev)]
            tres = [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                    torch.empty((nprob, k), dtype=torch.int64, device=dev),
                    torch.empty((nprob,), dtype=torch.int32, device=dev)]
            cnt = torch.zeros((nprob, ny * nx), dtype=torch.int32, device=dev)
            taken = torch.zeros(n, dtype=torch.bool, device=dev)
            P = 2 * R + 1
            win = torch.empty((n, P, P), dtype=torch.float64, device=dev)
            vv, uu = torch.meshgrid(torch.arange(P, device=dev) - R, torch.arange(P, device=dev) - R, indexing="ij")
            first = torch.arange(0, n, K, dtype=torch.int64, device=dev)
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        zero = torch.zeros((), dtype=torch.uint8, device=dev)
        w = dict(problems=nprob, candidates_per_problem=K, positions_per_problem=npos, headings=nhead, fov_deg=90,
                 nx=nx, ny=ny, radius=R, shape="disk", threshold=thr, k=k, m={})

        def run(m):
            return lambda: ctx.visibility_cover_greedy_view_batch_dev(
                occ_t, xy_t, v_t, ptr_t, k, m, thr, R, vhp.RANGE_DISK, pick_t=o[0], gain_t=o[1], npicked_t=o[2],
                count_t=o[3], weights_t=w_rand)

        def torch_windows(m):
            """m-fold greedy over view-masked window coverage S (n, P, P) at global cells `cell`"""
            ctx.visibility_window_batch_dev(occ_t, xy_t, R, win)
            sx, sy = xy_t[:, 0, None, None], xy_t[:, 1, None, None]
            x, y = sx + uu, sy + vv
            S = (x >= 0) & (x < nx) & (y >= 0) & (y < ny) & (win >= thr)
            S &= ~(((x == 0) & (sx != 0)) | ((y == 0) & (sy != 0)))
            r, ax, ay, bx, by = (v_t[:, i, None, None].long() for i in range(5))
            S &= uu * uu + vv * vv <= r * r
            c1, c2 = ax * vv - ay * uu, uu * by - vv * bx
            cab, dab = ax * by - ay * bx, ax * bx + ay * by
            inter, union = (c1 >= 0) & (c2 >= 0), (c1 >= 0) | (c2 >= 0)
            S &= torch.where(cab > 0, inter, torch.where((cab < 0) | (dab < 0), union, True)) | ((uu == 0) & (vv == 0))
            cell = gid[:, None, None].long() * (ny * nx) + y.clamp(0, ny - 1).long() * nx + x.clamp(0, nx - 1)
            wcell = w_rand.view(-1)[cell]
            pick, gain, npicked = tres
            pick.fill_(-1)
            gain.zero_()
            npicked.zero_()
            cnt.zero_()
            taken.zero_()
            flat = cnt.view(-1)
            for rd in range(k):
                live = S & (flat[cell] < m) & ~taken[:, None, None]
                gg = torch.where(live, wcell, zero).sum((1, 2), dtype=torch.int64)
                key = (gg << 28) | (IDX - kid.long())
                best = torch.zeros(nprob, dtype=torch.int64, device=dev).scatter_reduce_(0, gid.long(), key, "amax")
                act, bk = record_picks(torch, best, rd, tres)
                c = (first + torch.where(act, bk, 0)).clamp(max=n - 1)
                taken[c[act]] = True
                flat.scatter_add_(0, cell[c].view(-1), (S[c] & act[:, None, None]).view(-1).int())
                flat.clamp_(max=m)

        for m in (1, 2):
            d = dict(paths={})
            before = ctx.launches
            run(m)()
            ctx.synchronize()
            d["launches"] = ctx.launches - before
            d["paths"]["view"] = T(run(m))
            d["paths"]["torch"] = T(lambda: torch_windows(m))
            ctx.synchronize()
            run(m)()
            ctx.synchronize()
            d["torch_equals_view"] = bool(torch.equal(tres[0], o[0]) and torch.equal(tres[1], o[1]) and
                                          torch.equal(tres[2], o[2]) and
                                          torch.equal(cnt.view(nprob, ny, nx), o[3].int()))
            d["speedup"] = d["paths"]["torch"]["ms_median"] / d["paths"]["view"]["ms_median"]
            d["kernels_view"] = kernel_times(torch, ctx, run(m))
            d["npicked_total"] = int(o[2].sum().item())
            d["gain_total"] = int(o[1].sum().item())
            w["m"][str(m)] = d
            print(name, f"m={m}", json.dumps(d), flush=True)
        res["workloads"][name] = w
        del o, tres, cnt, taken, w_rand, win, xy_t, v_t
        torch.cuda.empty_cache()

    # omni: the m-fold call's g16384 with omnidirectional views
    R, k, m, n = 32, 256, 2, 65536
    xy = free_sources(g, occ16.cpu().numpy(), n)
    a = g.integers(-32767, 32768, (n, 2))
    a[(a == 0).all(1)] = (1, 0)
    views = np.concatenate([np.full((n, 1), R), a, a], 1).astype(np.int32)
    with torch.cuda.stream(stream):
        xy_t, v_t = torch.from_numpy(xy).to(dev), torch.from_numpy(views).to(dev)
        ptr_t = torch.tensor([0, n], dtype=torch.int64, device=dev)
        w_rand = weights(1, 16384, 16384)
        outs = [[torch.empty((1, k), dtype=torch.int32, device=dev), torch.empty((1, k), dtype=torch.int64, device=dev),
                 torch.empty((1,), dtype=torch.int32, device=dev),
                 torch.empty((1, 16384, 16384), dtype=torch.uint8, device=dev)] for _ in range(2)]
    stream.synchronize()
    ctx.prepare_maps_dev(occ16)

    def run_view():
        o = outs[0]
        ctx.visibility_cover_greedy_view_batch_dev(occ16, xy_t, v_t, ptr_t, k, m, thr, R, vhp.RANGE_DISK, pick_t=o[0],
                                                   gain_t=o[1], npicked_t=o[2], count_t=o[3], weights_t=w_rand)

    def run_mfold():
        o = outs[1]
        ctx.visibility_cover_greedy_mfold_batch_dev(occ16, xy_t, ptr_t, k, m, thr, R, vhp.RANGE_DISK, pick_t=o[0],
                                                    gain_t=o[1], npicked_t=o[2], count_t=o[3], weights_t=w_rand)

    d = dict(candidates=n, nx=16384, ny=16384, radius=R, shape="disk", threshold=thr, k=k, m=m, paths={})
    # alternate the two calls so that both see the same state of the machine
    tv, tm = [], []
    for _ in range(args.reps):
        tv.append(T(run_view)["ms_median"])
        tm.append(T(run_mfold)["ms_median"])
    d["paths"]["view"] = dict(ms_median=float(np.median(tv)), ms_min=min(tv), ms_max=max(tv), rounds=args.reps)
    d["paths"]["mfold"] = dict(ms_median=float(np.median(tm)), ms_min=min(tm), ms_max=max(tm), rounds=args.reps)
    run_view()
    run_mfold()
    ctx.synchronize()
    d["view_equals_mfold"] = bool(all(torch.equal(x, y) for x, y in zip(*outs)))
    d["view_cost"] = d["paths"]["view"]["ms_median"] / d["paths"]["mfold"]["ms_median"]
    d["kernels_view"] = kernel_times(torch, ctx, run_view)
    d["kernels_mfold"] = kernel_times(torch, ctx, run_mfold)
    d["candidate_bit_bytes"] = n * 65 * 3 * 4
    print("omni", json.dumps(d), flush=True)
    res["workloads"]["omni"] = d
    ctx.close()
    res["all_paths_equal"] = bool(d["view_equals_mfold"] and all(
        res["workloads"][nm]["m"][mm]["torch_equals_view"] for nm in ("cam16384", "cam1000") for mm in ("1", "2")))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
