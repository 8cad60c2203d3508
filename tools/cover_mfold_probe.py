"""Redundant (m-fold) greedy sensor placement (vhp_visibility_cover_greedy_mfold_batch_dev): device time on the three
workloads of cover_probe.py with a random importance map.  Prints one JSON line.

    python tools/cover_mfold_probe.py [--reps 5] [--warm 2] [--out FILE]

Per workload (maps packed once with prepare_maps_dev; threshold 0.5; the random uint8 weights of
cover_weighted_probe.py, a fifth of them 0):
  m = 1    the m-fold call against the weighted call (vhp_visibility_cover_greedy_weighted_batch_dev) on the same
           inputs, which must give the same picks, gains and npicked, and count > 0 equal to covered.  The difference
           is what the counters cost.
  m = 2, 3 the m-fold call against a torch m-fold greedy over the same candidate sets, built from fp64 windows
           (visibility_window_batch_dev), or on w1000 from whole-field bits (visibility_batch_bin_dev), recomputing
           every gain each round; pick, gain, npicked and count must be exactly equal.
`kernels` is the device time of one call per kernel (torch.profiler, a run of its own) for the weighted call and for
each m.  Times are CUDA events on the context's stream after warm-up: median, min and max over the repeats.
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
from cover_weighted_probe import IDX, record_picks  # noqa: E402
from merge_probe import free_sources, gpu_info, shipped_map, timed  # noqa: E402
from window_probe import obstacle_map  # noqa: E402


def kernel_times(torch, ctx, fn):
    """device time (us) and calls per kernel of one call of fn"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
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
    return kern


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("cover_mfold_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(13)
    res = dict(probe="cover_mfold", gpu=gpu_info(), workloads={})
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
        wrng = np.random.default_rng(29)
        wr = wrng.integers(0, 256, (nprob, ny, nx), dtype=np.uint8)
        wr[wrng.random((nprob, ny, nx)) < 0.2] = 0
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)
            gm_t = torch.arange(nprob, dtype=torch.int32, device=dev) if nmaps > 1 else None
            gid = torch.div(torch.arange(n, device=dev, dtype=torch.int32), K, rounding_mode="floor")
            kid = torch.arange(n, device=dev, dtype=torch.int32) % K
            w_rand = torch.from_numpy(wr).to(dev)
            o_w = [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                   torch.empty((nprob, k), dtype=torch.int64, device=dev),
                   torch.empty((nprob,), dtype=torch.int32, device=dev),
                   torch.empty((nprob, ny, nw), dtype=torch.int32, device=dev)]
            o_m = [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                   torch.empty((nprob, k), dtype=torch.int64, device=dev),
                   torch.empty((nprob,), dtype=torch.int32, device=dev),
                   torch.empty((nprob, ny, nx), dtype=torch.uint8, device=dev)]
        del wr
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)
        w = dict(problems=nprob, candidates_per_problem=K, maps=nmaps, nx=nx, ny=ny, radius=R,
                 shape="disk" if disk else "box", threshold=thr, k=k, rounds_enqueued=min(k, K), m={})

        def run_w():
            ctx.visibility_cover_greedy_weighted_batch_dev(occ_t, xy_t, ptr_t, k, thr, R, shape, pick_t=o_w[0],
                                                           gain_t=o_w[1], npicked_t=o_w[2], covered_t=o_w[3],
                                                           group_map_t=gm_t, weights_t=w_rand)

        def run_m(m):
            return lambda: ctx.visibility_cover_greedy_mfold_batch_dev(
                occ_t, xy_t, ptr_t, k, m, thr, R, shape, pick_t=o_m[0], gain_t=o_m[1], npicked_t=o_m[2],
                count_t=o_m[3], group_map_t=gm_t, weights_t=w_rand)

        # m = 1 against the weighted call
        d = dict(paths={})
        before = ctx.launches
        run_m(1)()
        ctx.synchronize()
        d["launches_mfold"] = ctx.launches - before
        d["paths"]["mfold"] = T(run_m(1))
        d["paths"]["weighted"] = T(run_w)
        run_w()
        run_m(1)()
        ctx.synchronize()
        d["weighted_equals_mfold"] = bool(
            torch.equal(o_w[0], o_m[0]) and torch.equal(o_w[1], o_m[1]) and torch.equal(o_w[2], o_m[2]) and
            torch.equal(unpack(torch, o_w[3], nx), o_m[3] > 0) and int(o_m[3].max().item()) <= 1)
        d["counter_cost"] = d["paths"]["mfold"]["ms_median"] / d["paths"]["weighted"]["ms_median"]
        d["kernels_weighted"] = kernel_times(torch, ctx, run_w)
        d["kernels_mfold"] = kernel_times(torch, ctx, run_m(1))
        w["m"]["1"] = d
        print(name, "m=1", json.dumps(d), flush=True)

        # m = 2, 3 against a torch m-fold greedy
        tres = [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                torch.empty((nprob, k), dtype=torch.int64, device=dev),
                torch.empty((nprob,), dtype=torch.int32, device=dev)]
        with torch.cuda.stream(stream):
            cnt = torch.zeros((nprob, ny * nx), dtype=torch.int32, device=dev)
            taken = torch.zeros(n, dtype=torch.bool, device=dev)
            if name != "w1000":
                P = 2 * R + 1
                win = torch.empty((n, P, P), dtype=torch.float64, device=dev)
                v, u = torch.meshgrid(torch.arange(P, device=dev) - R, torch.arange(P, device=dev) - R,
                                      indexing="ij")
                first = torch.arange(0, n, K, dtype=torch.int64, device=dev)
            else:
                bits = torch.empty((n, ny, nw), dtype=torch.int32, device=dev)
        stream.synchronize()
        zero = torch.zeros((), dtype=torch.uint8, device=dev)

        def reset():
            pick, gain, npicked = tres
            pick.fill_(-1)
            gain.zero_()
            npicked.zero_()
            cnt.zero_()
            taken.zero_()

        def torch_windows(m):
            """m-fold greedy over window coverage S (n, P, P) at global cells `cell`"""
            ctx.visibility_window_batch_dev(occ_t, xy_t, R, win)
            x = xy_t[:, 0, None, None] + u
            y = xy_t[:, 1, None, None] + v
            S = (x >= 0) & (x < nx) & (y >= 0) & (y < ny) & (win >= thr)
            if disk:
                S &= (u * u + v * v <= R * R)
            S &= ~(((x == 0) & (xy_t[:, 0, None, None] != 0)) | ((y == 0) & (xy_t[:, 1, None, None] != 0)))
            cell = gid[:, None, None].long() * (ny * nx) + y.clamp(0, ny - 1).long() * nx + x.clamp(0, nx - 1)
            wcell = w_rand.view(-1)[cell]
            reset()
            flat = cnt.view(-1)
            for r in range(k):
                live = S & (flat[cell] < m) & ~taken[:, None, None]
                gg = torch.where(live, wcell, zero).sum((1, 2), dtype=torch.int64)
                key = (gg << 28) | (IDX - kid.long())
                best = torch.zeros(nprob, dtype=torch.int64, device=dev).scatter_reduce_(0, gid.long(), key, "amax")
                act, bk = record_picks(torch, best, r, tres)
                c = (first + torch.where(act, bk, 0)).clamp(max=n - 1)
                taken[c[act]] = True
                flat.scatter_add_(0, cell[c].view(-1), (S[c] & act[:, None, None]).view(-1).int())
                flat.clamp_(max=m)

        per = max(1, (1 << 29) // (K * ny * nw * 32))  # problems per chunk of unpacked candidates

        def torch_bits(m):
            ctx.visibility_batch_bin_dev(occ_t, xy_t, thr, bits, src_map_t=gid)
            pick, gain, npicked = tres
            reset()
            for q0 in range(0, nprob, per):
                q1 = min(nprob, q0 + per)
                S = unpack(torch, bits[q0 * K:q1 * K], nx).reshape(q1 - q0, K, ny * nx)
                Wq = w_rand[q0:q1].reshape(q1 - q0, 1, ny * nx)
                Cq = cnt[q0:q1]
                tq = taken[q0 * K:q1 * K].view(q1 - q0, K)
                sub = [pick[q0:q1], gain[q0:q1], npicked[q0:q1]]
                ar = torch.arange(q1 - q0, device=dev)
                for r in range(k):
                    live = S & (Cq[:, None, :] < m) & ~tq[:, :, None]
                    gg = torch.where(live, Wq, zero).sum(2, dtype=torch.int64)
                    key = (gg << 28) | (IDX - torch.arange(K, device=dev)[None, :])
                    act, bk = record_picks(torch, key.max(1).values, r, sub)
                    c = torch.where(act, bk, 0)
                    tq[ar, c] |= act
                    Cq += (S[ar, c] & act[:, None]).int()
                    Cq.clamp_(max=m)
                del S

        for m in (2, 3):
            d = dict(paths={})
            d["paths"]["mfold"] = T(run_m(m))
            fn = (lambda: torch_bits(m)) if name == "w1000" else (lambda: torch_windows(m))
            d["paths"]["torch"] = T(fn)
            ctx.synchronize()
            run_m(m)()
            ctx.synchronize()
            d["torch_equals_mfold"] = bool(torch.equal(tres[0], o_m[0]) and torch.equal(tres[1], o_m[1]) and
                                           torch.equal(tres[2], o_m[2]) and
                                           torch.equal(cnt.view(nprob, ny, nx), o_m[3].int()))
            d["kernels_mfold"] = kernel_times(torch, ctx, run_m(m))
            d["npicked_total"] = int(o_m[2].sum().item())
            d["gain_total"] = int(o_m[1].sum().item())
            d["cells_at_m"] = int((o_m[3] == m).sum().item())
            w["m"][str(m)] = d
            print(name, f"m={m}", json.dumps(d), flush=True)
        res["workloads"][name] = w
        del occ_t, o_w, o_m, tres, cnt, taken, w_rand
        if name != "w1000":
            del win
        else:
            del bits
        torch.cuda.empty_cache()
    ctx.close()
    res["all_paths_equal"] = all(w["m"]["1"]["weighted_equals_mfold"] and w["m"]["2"]["torch_equals_mfold"] and
                                 w["m"]["3"]["torch_equals_mfold"] for w in res["workloads"].values())
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
