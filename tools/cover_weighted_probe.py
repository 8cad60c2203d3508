"""Weighted greedy sensor placement (vhp_visibility_cover_greedy_weighted_batch_dev): device time on the three
workloads of cover_probe.py under two weightings.  Prints one JSON line.

    python tools/cover_weighted_probe.py [--reps 5] [--warm 2] [--out FILE]

Weightings and what each is timed against (maps packed once with prepare_maps_dev; threshold 0.5):
  ones     every weight 1, passed as a weight tensor: the weighted call against the existing unweighted call
           (vhp_visibility_cover_greedy_batch_dev, no target) on the same inputs, which must give the same picks,
           npicked and covered, and the same gains as integers.  The difference is what the weights cost.
  random   a seeded uniform uint8 importance map per problem, a fifth of it 0: the weighted call against a torch
           weighted greedy over the same candidate sets, built from fp64 windows (visibility_window_batch_dev), or on
           w1000 from whole-field bits (visibility_batch_bin_dev), recomputing every gain each round.
Phases of the weighted call as cover_probe.py defines them: `sweep` is the call with k = 1 (the sweep, the weight plane,
the gains of round 0 and one pick); `greedy` is the rest, (total - sweep), over rounds - 1 rounds.  `kernels` is the
device time of one weighted call per kernel (torch.profiler, a run of its own).
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.  Each workload and
weighting records whether pick, gain, npicked and covered are exactly equal across its paths.
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

from cover_probe import unpack  # noqa: E402
from merge_probe import free_sources, gpu_info, shipped_map, timed  # noqa: E402
from window_probe import obstacle_map  # noqa: E402

IDX = 2**28 - 1  # index bits of the weighted key


def record_picks(torch, best, r, res):
    """record round r of every problem from its best key; returns (active, index within the group)"""
    pick, gain, npicked = res
    bg = best >> 28
    act = bg > 0
    bk = IDX - (best & IDX)
    pick[:, r] = torch.where(act, bk, -1).int()
    gain[:, r] = bg
    npicked += act.int()
    return act, bk


def torch_weighted_windows(torch, S, wcell, cell, gid, kid, nprob, k, res, U):
    """weighted greedy over window coverage S (n, W, W) bool at global cells `cell`, weights wcell (n, W, W) uint8"""
    pick, gain, npicked = res
    U.zero_()
    pick.fill_(-1)
    gain.zero_()
    npicked.zero_()
    gid64 = gid.long()
    first = torch.zeros(nprob, dtype=torch.int64, device=S.device).scatter_reduce_(
        0, gid64, torch.arange(S.shape[0], device=S.device), "amin", include_self=False)
    zero = torch.zeros((), dtype=torch.uint8, device=S.device)
    for r in range(k):
        g = torch.where(S & (U.view(-1)[cell] == 0), wcell, zero).sum((1, 2), dtype=torch.int64)
        key = (g << 28) | (IDX - kid.long())
        best = torch.zeros(nprob, dtype=torch.int64, device=S.device).scatter_reduce_(0, gid64, key, "amax")
        act, bk = record_picks(torch, best, r, res)
        c = (first + torch.where(act, bk, 0)).clamp(max=S.shape[0] - 1)
        m = S[c] & act[:, None, None]
        U.view(-1).scatter_reduce_(0, cell[c].view(-1), m.view(-1).to(torch.uint8), "amax")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("cover_weighted_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(13)
    res = dict(probe="cover_weighted", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731

    def shipped_maps(n):
        return torch.from_numpy(np.stack([shipped_map(g) for _ in range(n)])).to(dev)

    def workloads():  # those of cover_probe.py
        occ_t = obstacle_map(vhp, torch, dev, 16384, 16384)
        yield "g16384", occ_t, free_sources(g, occ_t.cpu().numpy(), 65536), 65536, 32, vhp.RANGE_DISK, 256
        occ_t = shipped_maps(1)
        yield "c1000", occ_t, free_sources(g, occ_t.cpu().numpy(), 256 * 64), 64, 64, vhp.RANGE_DISK, 8
        occ_t = shipped_maps(64)
        yield "w1000", occ_t, free_sources(g, occ_t.cpu().numpy(), 256), 256, 999, vhp.RANGE_BOX, 16

    thr = 0.5
    for name, occ_t, xy, K, R, shape, k in workloads():
        nmaps, ny, nx = occ_t.shape
        n, nw = xy.shape[0], (nx + 31) // 32
        nprob = n // K
        disk = shape == vhp.RANGE_DISK
        rounds = min(k, K)
        wrng = np.random.default_rng(29)
        wr = wrng.integers(0, 256, (nprob, ny, nx), dtype=np.uint8)
        wr[wrng.random((nprob, ny, nx)) < 0.2] = 0
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            gm_t = torch.arange(nprob, dtype=torch.int32, device=dev) if nmaps > 1 else None
            gid = torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
            kid = torch.arange(n, device=dev, dtype=torch.int32) % K
            w_ones = torch.ones((nprob, ny, nx), dtype=torch.uint8, device=dev)
            w_rand = torch.from_numpy(wr).to(dev)

            def outs(kk=k, gdt=torch.int64):
                return [torch.empty((nprob, kk), dtype=torch.int32, device=dev),
                        torch.empty((nprob, kk), dtype=gdt, device=dev),
                        torch.empty((nprob,), dtype=torch.int32, device=dev),
                        torch.empty((nprob, ny, nw), dtype=torch.int32, device=dev)]
            o_w, o_u = outs(), outs(gdt=torch.int32)
            o1 = outs(1)[:3] + [None]
        del wr
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        w = dict(problems=nprob, candidates_per_problem=K, maps=nmaps, nx=nx, ny=ny, radius=R,
                 shape="disk" if disk else "box", threshold=thr, k=k, rounds_enqueued=rounds, weightings={})

        def run_w(o, kk, wt):
            return lambda: ctx.visibility_cover_greedy_weighted_batch_dev(
                occ_t, xy_t, ptr_t, kk, thr, R, shape, pick_t=o[0], gain_t=o[1], npicked_t=o[2], covered_t=o[3],
                group_map_t=gm_t, weights_t=wt)

        def run_u(o):
            return lambda: ctx.visibility_cover_greedy_batch_dev(occ_t, xy_t, ptr_t, k, thr, R, shape, pick_t=o[0],
                                                                 gain_t=o[1], npicked_t=o[2], covered_t=o[3],
                                                                 group_map_t=gm_t)

        def weighted(wt):
            d = dict(paths={})
            before = ctx.launches
            run_w(o_w, k, wt)()
            ctx.synchronize()
            d["launches_weighted"] = ctx.launches - before
            d["paths"]["weighted"] = T(run_w(o_w, k, wt))
            sweep = T(run_w(o1, 1, wt))
            total = d["paths"]["weighted"]["ms_median"]
            d["phases_weighted"] = dict(sweep_ms=sweep["ms_median"], greedy_ms=total - sweep["ms_median"],
                                        us_per_round=1e3 * (total - sweep["ms_median"]) / max(rounds - 1, 1))
            return d

        # all ones against the unweighted call
        d = weighted(w_ones)
        d["paths"]["unweighted"] = T(run_u(o_u))
        run_w(o_w, k, w_ones)()
        run_u(o_u)()
        ctx.synchronize()
        d["unweighted_equals_weighted"] = bool(
            torch.equal(o_w[0], o_u[0]) and torch.equal(o_w[1], o_u[1].long()) and torch.equal(o_w[2], o_u[2]) and
            torch.equal(o_w[3], o_u[3]))
        d["weight_cost"] = d["paths"]["weighted"]["ms_median"] / d["paths"]["unweighted"]["ms_median"]
        w["weightings"]["ones"] = d
        print(name, "ones", json.dumps(d), flush=True)

        # a random importance map against a torch weighted greedy
        d = weighted(w_rand)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_w(o_w, k, w_rand)()
            ctx.synchronize()
        kern = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = getattr(e, "cuda_time_total", 0)
            if t and "Memset" not in e.key and "Memcpy" not in e.key:
                kname = e.key.replace("(anonymous namespace)::", "").split("(")[0].split("::")[-1]
                acc = kern.setdefault(kname, dict(us=0.0, calls=0))
                acc["us"] += t
                acc["calls"] += e.count
        d["kernels"] = kern
        tres = [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                torch.empty((nprob, k), dtype=torch.int64, device=dev),
                torch.empty((nprob,), dtype=torch.int32, device=dev)]
        if name != "w1000":
            W = 2 * R + 1
            with torch.cuda.stream(stream):
                win = torch.empty((n, W, W), dtype=torch.float64, device=dev)
                v, u = torch.meshgrid(torch.arange(W, device=dev) - R, torch.arange(W, device=dev) - R, indexing="ij")
                U = torch.zeros((nprob, ny, nx), dtype=torch.uint8, device=dev)
            stream.synchronize()

            def torch_path():
                ctx.visibility_window_batch_dev(occ_t, xy_t, R, win)
                x = xy_t[:, 0, None, None] + u
                y = xy_t[:, 1, None, None] + v
                S = (x >= 0) & (x < nx) & (y >= 0) & (y < ny) & (win >= thr)
                if disk:
                    S &= (u * u + v * v <= R * R)
                S &= ~(((x == 0) & (xy_t[:, 0, None, None] != 0)) | ((y == 0) & (xy_t[:, 1, None, None] != 0)))
                cell = gid[:, None, None].long() * (ny * nx) + y.clamp(0, ny - 1).long() * nx + x.clamp(0, nx - 1)
                wcell = w_rand.view(-1)[cell]
                torch_weighted_windows(torch, S, wcell, cell, gid, kid, nprob, k, tres, U)
            d["paths"]["torch"] = T(torch_path)
            ctx.synchronize()
            Ub = U.bool()
            del win
        else:
            with torch.cuda.stream(stream):
                bits = torch.empty((n, ny, nw), dtype=torch.int32, device=dev)
                Ub = torch.zeros((nprob, ny * nx), dtype=torch.bool, device=dev)
            stream.synchronize()
            per = max(1, (1 << 29) // (K * ny * nw * 32))  # problems per chunk of unpacked candidates
            zero = torch.zeros((), dtype=torch.uint8, device=dev)

            def torch_path():
                ctx.visibility_batch_bin_dev(occ_t, xy_t, thr, bits, src_map_t=gid)
                pick, gain, npicked = tres
                pick.fill_(-1)
                gain.zero_()
                npicked.zero_()
                Ub.zero_()
                for q0 in range(0, nprob, per):
                    q1 = min(nprob, q0 + per)
                    S = unpack(torch, bits[q0 * K:q1 * K], nx).reshape(q1 - q0, K, ny * nx)
                    Wq = w_rand[q0:q1].reshape(q1 - q0, 1, ny * nx)
                    Uq = Ub[q0:q1]
                    sub = [pick[q0:q1], gain[q0:q1], npicked[q0:q1]]
                    for r in range(k):
                        gg = torch.where(S & ~Uq[:, None, :], Wq, zero).sum(2, dtype=torch.int64)
                        key = (gg << 28) | (IDX - torch.arange(K, device=dev)[None, :])
                        act, bk = record_picks(torch, key.max(1).values, r, sub)
                        Uq |= S[torch.arange(q1 - q0, device=dev), torch.where(act, bk, 0)] & act[:, None]
                    del S
            d["paths"]["torch"] = T(torch_path)
            ctx.synchronize()
            Ub = Ub.view(nprob, ny, nx)
            del bits
        run_w(o_w, k, w_rand)()
        ctx.synchronize()
        cov = unpack(torch, o_w[3], nx)
        d["torch_equals_weighted"] = bool(torch.equal(tres[0], o_w[0]) and torch.equal(tres[1], o_w[1]) and
                                          torch.equal(tres[2], o_w[2]) and torch.equal(Ub, cov))
        d["npicked_total"] = int(o_w[2].sum().item())
        d["gain_total"] = int(o_w[1].sum().item())
        d["covered_cells"] = int(cov.sum().item())
        w["weightings"]["random"] = d
        print(name, "random", json.dumps(d), flush=True)
        res["workloads"][name] = w
        del occ_t, o_w, o_u, o1, tres, Ub, cov, w_ones, w_rand
        torch.cuda.empty_cache()
    ctx.close()
    res["all_paths_equal"] = all(w["weightings"]["ones"]["unweighted_equals_weighted"] and
                                 w["weightings"]["random"]["torch_equals_weighted"]
                                 for w in res["workloads"].values())
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
