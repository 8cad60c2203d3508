"""Budgeted sensor placement (vhp_visibility_cover_budget_batch_dev): device time of mixed-fleet placement under a
budget, and what the 128-bit ratio key and the device loop cost against the calls it generalises.  Prints one JSON line.

    python tools/cover_budget_probe.py [--reps 5] [--warm 2] [--out FILE]

Workloads (maps packed once with prepare_maps_dev; threshold 0.5; disk ranges):
  fleet16384  cover_probe.py's 16384^2 map, 8192 free positions, each with 8 camera headings of 90 degrees and r = 24
              (cost 1) and one omnidirectional lidar of r = 32 (cost 4): 73 728 candidates in one problem, R = 32,
              random uint8 weights with a fifth of them 0, m = 1, budgets of 64, 256 and 1024 units.  Against a torch
              cost-benefit greedy over view-masked fp64 windows (cover_view_probe.py's baseline) that recomputes every
              gain each round and takes the argmax of the fp64 ratio gain / cost: with costs <= 8 and gains < 2^28 two
              distinct ratios differ by more than 2^-34 of their size, and equal ratios give equal doubles, so that
              baseline is an exact reference here (it is not in general: tests/test_cover_budget_cpu.py).
  unit_cam16384  cover_view_probe.py's cam16384 (8192 positions x 8 headings, R = 32, those weights) with every cost 1
              and a budget of 256, against the view call with k = 256: the same picks, so the difference is the price
              of the 128-bit key and the device loop.
  unit_g16384  cover_quota_probe.py's g16384 (65 536 omnidirectional candidates, every cell weighs 1) with every cost 1,
              budget UINT64_MAX and a quota of 50 % of the coverable total, against the quota call with that quota.
  fleet1000   256 problems x 16 positions x (4 cameras of 90 degrees, r = 48, cost 1 + 1 lidar, r = 64, cost 3) on the
              shipped-settings 1000^2 map, R = 64, those weights, budget 12, against the torch greedy.
Every pair of paths must give exactly equal pick, gain, npicked and count (and spent, against the torch greedy).
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.  `per_round_us` is
a path's median time over its largest npicked.  `kernels` is the device time per kernel of one call of the slowest
budget case (torch.profiler, a run of its own).
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
from merge_probe import free_sources, gpu_info, shipped_map, timed  # noqa: E402
from window_probe import obstacle_map  # noqa: E402

U64_MAX = np.iinfo(np.uint64).max
IDX = 2**28 - 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("cover_budget_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(23)
    res = dict(probe="cover_budget", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731
    thr = 0.5
    occ16 = obstacle_map(vhp, torch, dev, 16384, 16384)
    occ1 = torch.from_numpy(shipped_map(g)[None]).to(dev)
    all_equal = True
    drawn = {}  # each fleet workload's candidates, for the profile run

    def weights(nprob, ny, nx):
        wrng = np.random.default_rng(29)
        wr = wrng.integers(0, 256, (nprob, ny, nx), dtype=np.uint8)
        wr[wrng.random((nprob, ny, nx)) < 0.2] = 0
        return torch.from_numpy(wr).to(dev)

    def fleet(occ_t, nprob, npos, nhead, r_cam, r_lidar, c_cam, c_lidar):
        """per position nhead cameras of 90 degrees then one lidar, position-major"""
        pos = free_sources(g, occ_t.cpu().numpy(), nprob * npos)
        xy = np.repeat(pos, nhead + 1, axis=0)
        heads = np.arange(nhead) * (360.0 / nhead)
        cams = vhp.sensor_views(heads, 90, r_cam)
        lidar = np.array([[r_lidar, 1, 0, 1, 0]], np.int32)
        views = np.tile(np.concatenate([cams, lidar]), (nprob * npos, 1)).astype(np.int32)
        cost = np.tile(np.array([c_cam] * nhead + [c_lidar], np.uint32), nprob * npos)
        return xy, views, cost

    def outs(nprob, k, ny, nx):
        return dict(pick=torch.empty((nprob, k), dtype=torch.int32, device=dev),
                    gain=torch.empty((nprob, k), dtype=torch.int64, device=dev),
                    npicked=torch.empty((nprob,), dtype=torch.int32, device=dev),
                    count=torch.empty((nprob, ny, nx), dtype=torch.uint8, device=dev),
                    total=torch.empty((nprob,), dtype=torch.int64, device=dev),
                    spent=torch.empty((nprob,), dtype=torch.int64, device=dev),
                    single=torch.empty((nprob,), dtype=torch.int32, device=dev),
                    single_gain=torch.empty((nprob,), dtype=torch.int64, device=dev))

    def budget_fn(occ_t, xy_t, v_t, ptr_t, c_t, b_t, kmax, R, w_t, o, q_t=None):
        return lambda: ctx.visibility_cover_budget_batch_dev(
            occ_t, xy_t, ptr_t, c_t, b_t, kmax, thr, R, vhp.RANGE_DISK, quota_t=q_t, m=1, weights_t=w_t, views_t=v_t,
            **{k + "_t": v for k, v in o.items()})

    def torch_greedy(occ_t, xy_t, v_t, c_t, budget, nprob, K, R, w_t, kmax, tres):
        """cost-benefit greedy over view-masked fp64 windows: every gain recomputed each round, argmax of the fp64
        ratio among the affordable candidates of positive gain, ties to the smallest index"""
        _, ny, nx = occ_t.shape
        n = xy_t.shape[0]
        P = 2 * R + 1
        win = torch.empty((n, P, P), dtype=torch.float64, device=dev)
        ctx.visibility_window_batch_dev(occ_t, xy_t, R, win)
        vv, uu = torch.meshgrid(torch.arange(P, device=dev) - R, torch.arange(P, device=dev) - R, indexing="ij")
        gid = torch.div(torch.arange(n, device=dev), K, rounding_mode="floor")
        kid = torch.arange(n, device=dev) % K
        first = torch.arange(0, n, K, dtype=torch.int64, device=dev)
        sx, sy = xy_t[:, 0, None, None], xy_t[:, 1, None, None]
        x, y = sx + uu, sy + vv
        S = (x >= 0) & (x < nx) & (y >= 0) & (y < ny) & (win >= thr)
        del win
        S &= ~(((x == 0) & (sx != 0)) | ((y == 0) & (sy != 0)))
        r, ax, ay, bx, by = (v_t[:, i, None, None].long() for i in range(5))
        S &= uu * uu + vv * vv <= r * r
        c1, c2 = ax * vv - ay * uu, uu * by - vv * bx
        cab, dab = ax * by - ay * bx, ax * bx + ay * by
        inter, union = (c1 >= 0) & (c2 >= 0), (c1 >= 0) | (c2 >= 0)
        S &= torch.where(cab > 0, inter, torch.where((cab < 0) | (dab < 0), union, True)) | ((uu == 0) & (vv == 0))
        cell = gid[:, None, None] * (ny * nx) + y.clamp(0, ny - 1).long() * nx + x.clamp(0, nx - 1)
        wcell = w_t.view(-1)[cell]
        cost = c_t.long()
        costf = cost.double()
        pick, gain, npicked, spent, cnt = tres
        pick.fill_(-1)
        gain.zero_()
        npicked.zero_()
        spent.zero_()
        cnt.zero_()
        flat = cnt.view(-1)
        taken = torch.zeros(n, dtype=torch.bool, device=dev)
        left = torch.full((nprob,), budget, dtype=torch.int64, device=dev)
        zero = torch.zeros((), dtype=torch.uint8, device=dev)
        for rd in range(kmax):
            live = S & (flat[cell] < 1) & ~taken[:, None, None]
            gg = torch.where(live, wcell, zero).sum((1, 2), dtype=torch.int64)
            ok = (gg > 0) & (cost <= left[gid])
            ratio = torch.where(ok, gg.double() / costf, -1.0)
            best = torch.full((nprob,), -1.0, dtype=torch.float64, device=dev).scatter_reduce_(0, gid, ratio, "amax")
            tie = ok & (ratio == best[gid])
            bk = torch.full((nprob,), -1, dtype=torch.int64, device=dev).scatter_reduce_(
                0, gid, torch.where(tie, IDX - kid, -1), "amax")
            act = bk >= 0
            if not bool(act.any()):
                break
            k = IDX - bk
            c = (first + torch.where(act, k, 0)).clamp(max=n - 1)
            pick[:, rd] = torch.where(act, k, -1).int()
            gain[:, rd] = torch.where(act, gg[c], 0)
            npicked += act.int()
            spent += torch.where(act, cost[c], 0)
            left -= torch.where(act, cost[c], 0)
            taken[c[act]] = True
            flat.scatter_add_(0, cell[c].view(-1), (S[c] & act[:, None, None]).view(-1).int())
            flat.clamp_(max=1)

    def same(o, ref, keys):
        ok = True
        for key in keys:
            a, b = o[key], ref[key]
            ok &= bool(torch.equal(a.long(), b.long()))
        return ok

    def fleet_workload(name, occ_t, nprob, npos, nhead, r_cam, r_lidar, c_lidar, R, budgets):
        nonlocal all_equal
        _, ny, nx = occ_t.shape
        xy, views, cost = drawn[name] = fleet(occ_t, nprob, npos, nhead, r_cam, r_lidar, 1, c_lidar)
        n = xy.shape[0]
        K = n // nprob
        with torch.cuda.stream(stream):
            xy_t, v_t = torch.from_numpy(xy).to(dev), torch.from_numpy(views).to(dev)
            c_t = torch.from_numpy(cost.view(np.int32)).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            w_t = weights(nprob, ny, nx)
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        w = dict(problems=nprob, candidates_per_problem=K, positions_per_problem=npos,
                 cameras=dict(headings=nhead, fov_deg=90, r=r_cam, cost=1), lidar=dict(r=r_lidar, cost=c_lidar),
                 nx=nx, ny=ny, radius=R, shape="disk", threshold=thr, m=1, budgets={})
        for B in budgets:
            kmax = min(K, B)
            with torch.cuda.stream(stream):
                b_t = torch.full((nprob,), B, dtype=torch.int64, device=dev)
                o = outs(nprob, kmax, ny, nx)
                tres = [torch.empty((nprob, kmax), dtype=torch.int32, device=dev),
                        torch.empty((nprob, kmax), dtype=torch.int64, device=dev),
                        torch.empty((nprob,), dtype=torch.int32, device=dev),
                        torch.empty((nprob,), dtype=torch.int64, device=dev),
                        torch.zeros((nprob, ny * nx), dtype=torch.int32, device=dev)]
            fn = budget_fn(occ_t, xy_t, v_t, ptr_t, c_t, b_t, kmax, R, w_t, o)
            d = dict(kmax=kmax, paths={})
            before = ctx.launches
            fn()
            ctx.synchronize()
            d["launches"] = ctx.launches - before
            d["paths"]["budget"] = T(fn)
            d["paths"]["torch"] = T(lambda: torch_greedy(occ_t, xy_t, v_t, c_t, B, nprob, K, R, w_t, kmax, tres))
            fn()
            ctx.synchronize()
            ref = dict(pick=tres[0], gain=tres[1], npicked=tres[2], spent=tres[3],
                       count=tres[4].view(nprob, ny, nx))
            d["torch_equals_budget"] = same(o, ref, ("pick", "gain", "npicked", "spent", "count"))
            all_equal &= d["torch_equals_budget"]
            rounds = int(o["npicked"].max().item())
            d["rounds"] = rounds
            d["npicked_total"] = int(o["npicked"].sum().item())
            d["spent_total"] = int(o["spent"].sum().item())
            d["total"] = int(o["total"].sum().item())
            d["lidars_picked"] = int(sum((p % (nhead + 1) == nhead) for p in o["pick"].cpu().numpy().ravel() if p >= 0))
            d["best_single_count"] = int((o["single_gain"] > o["total"]).sum().item())
            d["per_round_us"] = 1e3 * d["paths"]["budget"]["ms_median"] / max(rounds, 1)
            d["speedup"] = d["paths"]["torch"]["ms_median"] / d["paths"]["budget"]["ms_median"]
            print(name, f"B={B}", json.dumps(d), flush=True)
            w["budgets"][str(B)] = d
            del o, tres
        res["workloads"][name] = w
        del xy_t, v_t, c_t, w_t
        torch.cuda.empty_cache()

    fleet_workload("fleet16384", occ16, 1, 8192, 8, 24, 32, 4, 32, (64, 256, 1024))
    fleet_workload("fleet1000", occ1, 256, 16, 4, 48, 64, 3, 64, (12,))

    # unit costs against the view call (cam16384, budget 256 = k) and the quota call (g16384, quota 50 %)
    ctx.prepare_maps_dev(occ16)
    R, n = 32, 65536
    pos = free_sources(g, occ16.cpu().numpy(), 8192)
    cam_xy = np.repeat(pos, 8, axis=0)
    cam_v = vhp.sensor_views(np.tile(np.arange(8) * 45.0, 8192), 90, R)
    g_xy = free_sources(g, occ16.cpu().numpy(), n)
    for name, xy, views, k in (("unit_cam16384", cam_xy, cam_v, 256), ("unit_g16384", g_xy, None, n)):
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            v_t = None if views is None else torch.from_numpy(views).to(dev)
            ptr_t = torch.tensor([0, n], dtype=torch.int64, device=dev)
            c_t = torch.ones((n,), dtype=torch.int32, device=dev)
            w_t = weights(1, 16384, 16384) if views is not None else None
            o = outs(1, k, 16384, 16384)
            ro = outs(1, k, 16384, 16384)
        stream.synchronize()
        d = dict(candidates=n, radius=R, shape="disk", threshold=thr, m=1, paths={})
        if views is not None:
            b_t = torch.full((1,), 256, dtype=torch.int64, device=dev)
            q_t = None
            d.update(views="90 degree cameras", budget=256, weights="random, a fifth 0")

            def ref():
                ctx.visibility_cover_greedy_view_batch_dev(occ16, xy_t, v_t, ptr_t, k, 1, thr, R, vhp.RANGE_DISK,
                                                           pick_t=ro["pick"], gain_t=ro["gain"],
                                                           npicked_t=ro["npicked"], count_t=ro["count"],
                                                           weights_t=w_t)
            ref_name = "view"
        else:
            b_t = torch.from_numpy(np.array([U64_MAX], np.uint64).view(np.int64)).to(dev)
            qall = torch.from_numpy(np.array([U64_MAX], np.uint64).view(np.int64)).to(dev)
            ctx.visibility_cover_quota_batch_dev(occ16, xy_t, ptr_t, qall, k, thr, R, vhp.RANGE_DISK,
                                                 total_t=ro["total"])
            ctx.synchronize()
            coverable = int(ro["total"].item())
            q_t = torch.tensor([(coverable + 1) // 2], dtype=torch.int64, device=dev)
            d.update(views=None, budget="UINT64_MAX", quota=int(q_t.item()), coverable_total=coverable)

            def ref():
                ctx.visibility_cover_quota_batch_dev(occ16, xy_t, ptr_t, q_t, k, thr, R, vhp.RANGE_DISK,
                                                     pick_t=ro["pick"], gain_t=ro["gain"], npicked_t=ro["npicked"],
                                                     count_t=ro["count"], total_t=ro["total"])
            ref_name = "quota"
        fn = budget_fn(occ16, xy_t, v_t, ptr_t, c_t, b_t, k, R, w_t, o, q_t)
        before = ctx.launches
        fn()
        ctx.synchronize()
        d["launches"] = ctx.launches - before
        before = ctx.launches
        ref()
        ctx.synchronize()
        d["launches_" + ref_name] = ctx.launches - before
        # alternate the two paths, twice, so a drift of the clocks shows as a spread
        for _ in range(2):
            for key, f in (("budget", fn), (ref_name, ref)):
                t = T(f)
                if key not in d["paths"] or t["ms_median"] < d["paths"][key]["ms_median"]:
                    d["paths"][key] = t
        fn()
        ref()
        ctx.synchronize()
        keys = ("pick", "gain", "npicked", "count") + (("total",) if views is None else ())
        d[ref_name + "_equals_budget"] = same(o, ro, keys)
        all_equal &= d[ref_name + "_equals_budget"]
        rounds = int(o["npicked"].max().item())
        d["rounds"] = rounds
        d["per_round_us"] = {p: 1e3 * t["ms_median"] / rounds for p, t in d["paths"].items()}
        d["budget_over_" + ref_name] = d["paths"]["budget"]["ms_median"] / d["paths"][ref_name]["ms_median"]
        d["kernels_budget"] = kernel_times(torch, ctx, fn)
        d["kernels_" + ref_name] = kernel_times(torch, ctx, ref)
        print(name, json.dumps(d), flush=True)
        res["workloads"][name] = d
        del o, ro, xy_t, v_t, c_t, w_t
        torch.cuda.empty_cache()

    # the slowest fleet case, per kernel
    slow = max(((nm, b) for nm in ("fleet16384", "fleet1000") for b in res["workloads"][nm]["budgets"]),
               key=lambda t: res["workloads"][t[0]]["budgets"][t[1]]["paths"]["budget"]["ms_median"])
    res["slowest"] = dict(workload=slow[0], budget=int(slow[1]))
    occ_t, nprob, R = (occ16, 1, 32) if slow[0] == "fleet16384" else (occ1, 256, 64)
    xy, views, cost = drawn[slow[0]]
    _, ny, nx = occ_t.shape
    n = xy.shape[0]
    B = int(slow[1])
    with torch.cuda.stream(stream):
        xy_t, v_t = torch.from_numpy(xy).to(dev), torch.from_numpy(views).to(dev)
        c_t = torch.from_numpy(cost.view(np.int32)).to(dev)
        ptr_t = torch.arange(0, n + 1, n // nprob, dtype=torch.int64, device=dev)
        w_t = weights(nprob, ny, nx)
        b_t = torch.full((nprob,), B, dtype=torch.int64, device=dev)
        o = outs(nprob, min(n // nprob, B), ny, nx)
    stream.synchronize()
    ctx.prepare_maps_dev(occ_t)
    fn = budget_fn(occ_t, xy_t, v_t, ptr_t, c_t, b_t, min(n // nprob, B), R, w_t, o)
    fn()
    ctx.synchronize()
    res["slowest"]["kernels"] = kernel_times(torch, ctx, fn)
    res["slowest"]["rounds"] = int(o["npicked"].max().item())
    ctx.close()
    res["all_paths_equal"] = bool(all_equal)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
