"""Greedy sensor placement (vhp_visibility_cover_greedy_batch_dev): device time of the direct route against the
fallback and against what callers write without the call, on three workloads.  Prints one JSON line.

    python tools/cover_probe.py [--reps 5] [--warm 2] [--out FILE]

Paths (the maps are packed once with prepare_maps_dev, as a caller with fixed maps would; threshold 0.5):
  direct     the sweep of each candidate's box writes its coverage bits (kFmtCoverBits), then the greedy rounds
  fallback   the same call with grid mode forced (set_grid_sweep(2)): the whole fields of the grid kernels, cropped to
             windows or, where a window would be larger than the map, kept whole, thresholded into the bits by
             cover_fold_kernel (not run on g16384: 65 536 sweeps of the whole 16384^2 map)
  torch      fp64 windows (visibility_window_batch_dev; w1000: visibility_batch_bin_dev whole-field bits), thresholded
             and masked in torch, and a torch greedy loop that recomputes every gain each round
Phases of the direct route: `sweep` is the call with k = 1 (the sweep, the gains of round 0 and one pick); `greedy` is
the rest of the call, (total - sweep), over rounds - 1 rounds.  `kernels` is the device time of one call per kernel
(torch.profiler, a run of its own): where the greedy kernels' busy time is far below the greedy phase, the rounds are
bound by launches, not by work.
Workloads:
  g16384  one problem of 65 536 disk candidates, R = 32, on the device-generated 16384 x 16384 map of
          merge_range_probe, k = 256 (the candidate bits, 65 536 x 65 rows x 3 words = 51 MB, fit in the 126 MB L2)
  c1000   256 problems x 64 disk candidates, R = 64, on one shipped-settings 1000 x 1000 map, k = 8
  w1000   box, R = 999: 64 problems x 256 candidates, one shipped-settings 1000 x 1000 map per problem, k = 16
Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.  Each workload
records whether pick, gain, npicked and covered are exactly equal across the paths.
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

KEY_LO = 2**31 - 1


def torch_greedy_windows(torch, S, cell, gid, kid, nprob, plane, k, res):
    """greedy over window coverage S (n, W, W) bool at global cells `cell` (problem * plane + y * nx + x)"""
    pick, gain, npicked, U = res
    U.zero_()
    pick.fill_(-1)
    gain.zero_()
    npicked.zero_()
    gid64 = gid.long()
    first = torch.zeros(nprob, dtype=torch.int64, device=S.device).scatter_reduce_(
        0, gid64, torch.arange(S.shape[0], device=S.device), "amin", include_self=False)
    for r in range(k):
        g = (S & (U.view(-1)[cell] == 0)).sum((1, 2))
        key = (g << 32) | (KEY_LO - kid.long())
        best = torch.zeros(nprob, dtype=torch.int64, device=S.device).scatter_reduce_(0, gid64, key, "amax")
        bg = best >> 32
        act = bg > 0
        bk = KEY_LO - (best & 0xffffffff)
        pick[:, r] = torch.where(act, bk, -1).int()
        gain[:, r] = bg.int()
        npicked += act.int()
        c = (first + torch.where(act, bk, 0)).clamp(max=S.shape[0] - 1)
        m = S[c] & act[:, None, None]
        U.view(-1).scatter_reduce_(0, cell[c].view(-1), m.view(-1).to(torch.uint8), "amax")


def unpack(torch, bits, nx):
    """int32 (..., nw) -> bool (..., nx)"""
    sh = torch.arange(32, device=bits.device, dtype=torch.int32)
    b = ((bits[..., None] >> sh) & 1).bool()
    return b.reshape(*bits.shape[:-1], bits.shape[-1] * 32)[..., :nx]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("cover_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(13)
    res = dict(probe="cover", gpu=gpu_info(), workloads={},
               note="g16384's candidate bits (65 536 x 65 x 3 words, 51 MB) fit in the B200's 126 MB L2")
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731

    def shipped_maps(n):
        return torch.from_numpy(np.stack([shipped_map(g) for _ in range(n)])).to(dev)

    def workloads():
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
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            gm_t = torch.arange(nprob, dtype=torch.int32, device=dev) if nmaps > 1 else None
            gid = torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
            kid = torch.arange(n, device=dev, dtype=torch.int32) % K

            def outs():
                return [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                        torch.empty((nprob, k), dtype=torch.int32, device=dev),
                        torch.empty((nprob,), dtype=torch.int32, device=dev),
                        torch.empty((nprob, ny, nw), dtype=torch.int32, device=dev)]
            o_direct, o_fb = outs(), outs()
            o1 = outs()[:3] + [None]
            o1[0] = torch.empty((nprob, 1), dtype=torch.int32, device=dev)
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        rounds = min(k, K)
        w = dict(problems=nprob, candidates_per_problem=K, maps=nmaps, nx=nx, ny=ny, radius=R,
                 shape="disk" if disk else "box", threshold=thr, k=k, rounds_enqueued=rounds, paths={})

        def run(o, kk):
            return lambda: ctx.visibility_cover_greedy_batch_dev(occ_t, xy_t, ptr_t, kk, thr, R, shape, pick_t=o[0],
                                                                 gain_t=o[1], npicked_t=o[2], covered_t=o[3],
                                                                 group_map_t=gm_t)

        before = ctx.launches
        run(o_direct, k)()
        ctx.synchronize()
        w["launches_direct"] = ctx.launches - before
        w["paths"]["direct"] = T(run(o_direct, k))
        sweep = T(run(o1, 1))
        total = w["paths"]["direct"]["ms_median"]
        w["phases_direct"] = dict(sweep_ms=sweep["ms_median"], greedy_ms=total - sweep["ms_median"],
                                  us_per_round=1e3 * (total - sweep["ms_median"]) / max(rounds - 1, 1))
        if name == "g16384":
            w["fallback"] = "not run: forced grid mode sweeps the whole 16384 x 16384 map once per candidate"
        else:
            ctx.set_grid_sweep(2)
            before = ctx.launches
            run(o_fb, k)()
            ctx.synchronize()
            w["launches_fallback"] = ctx.launches - before
            w["paths"]["fallback"] = timed(torch, stream, run(o_fb, k), args.reps, 1)
            ctx.set_grid_sweep(1)
            run(o_direct, k)()
            ctx.synchronize()
            w["fallback_equals_direct"] = bool(all(torch.equal(a, b) for a, b in zip(o_direct, o_fb)))
        del o_fb

        # per-kernel device time of one direct call
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(o_direct, k)()
            ctx.synchronize()
        kern = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = getattr(e, "cuda_time_total", 0)
            if t and "Memset" not in e.key and "Memcpy" not in e.key:
                kname = e.key.replace("(anonymous namespace)::", "").split("(")[0].split("<")[0].split("::")[-1]
                acc = kern.setdefault(kname, dict(us=0.0, calls=0))
                acc["us"] += t
                acc["calls"] += e.count
        w["kernels"] = kern
        busy = sum(v["us"] for kname, v in kern.items() if kname.startswith("cover_") and "fold" not in kname)
        w["greedy_kernels_busy_ms"] = busy / 1e3
        w["greedy_launch_bound"] = bool(busy / 1e3 < 0.5 * w["phases_direct"]["greedy_ms"])

        # what callers write today
        tres = [torch.empty((nprob, k), dtype=torch.int32, device=dev), torch.empty((nprob, k), dtype=torch.int32,
                device=dev), torch.empty((nprob,), dtype=torch.int32, device=dev)]
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
                torch_greedy_windows(torch, S, cell, gid, kid, nprob, ny * nx, k, tres + [U])
            w["paths"]["torch"] = T(torch_path)
            ctx.synchronize()
            Ub = U.bool()
            del win
        else:
            with torch.cuda.stream(stream):
                bits = torch.empty((n, ny, nw), dtype=torch.int32, device=dev)
                Ub = torch.zeros((nprob, ny * nx), dtype=torch.bool, device=dev)
            stream.synchronize()
            per = max(1, (1 << 29) // (K * ny * nw * 32))  # problems per chunk of unpacked candidates

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
                    Uq = Ub[q0:q1]
                    for r in range(k):
                        gg = (S & ~Uq[:, None, :]).sum(2)
                        key = (gg << 32) | (KEY_LO - torch.arange(K, device=dev)[None, :])
                        best = key.max(1).values
                        bg = best >> 32
                        act = bg > 0
                        bk = KEY_LO - (best & 0xffffffff)
                        pick[q0:q1, r] = torch.where(act, bk, -1).int()
                        gain[q0:q1, r] = bg.int()
                        npicked[q0:q1] += act.int()
                        sel = S[torch.arange(q1 - q0, device=dev), torch.where(act, bk, 0)] & act[:, None]
                        Uq |= sel
                    del S
            w["paths"]["torch"] = T(torch_path)
            ctx.synchronize()
            Ub = Ub.view(nprob, ny, nx)
            del bits
        cov = unpack(torch, o_direct[3], nx)
        w["torch_equals_direct"] = bool(torch.equal(tres[0], o_direct[0]) and torch.equal(tres[1], o_direct[1]) and
                                        torch.equal(tres[2], o_direct[2]) and torch.equal(Ub, cov))
        w["npicked_total"] = int(o_direct[2].sum().item())
        w["covered_cells"] = int(cov.sum().item())
        w["candidate_bits_bytes"] = n * min(2 * R + 1, ny) * min(nw, (2 * R + 31) // 32 + 1) * 4
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        del occ_t, o_direct, tres, Ub, cov
        torch.cuda.empty_cache()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
