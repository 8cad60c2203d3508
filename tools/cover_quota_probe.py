"""Quota sensor placement (vhp_visibility_cover_quota_batch_dev): device time of the fewest greedy picks that reach a
coverage quota, against the ways a caller gets the same answer from the fixed-k calls.  Prints one JSON line.

    python tools/cover_quota_probe.py [--reps 5] [--warm 2] [--out FILE]

Workloads (maps packed once with prepare_maps_dev; threshold 0.5; every cell weighs 1; R = 32 disk on 16384^2,
R = 64 disk on 1000^2):
  g16384 m1 / m2  cover_probe.py's g16384: one problem of 65 536 free candidates on the 16384^2 map, m = 1 and 2
  cam16384        cover_view_probe.py's cam16384: 8192 positions x 8 headings of 90 degrees, one problem, m = 1
  c1000           cover_probe.py's c1000: 256 problems x 64 candidates on one 1000^2 map, m = 1
  cam1000         cover_view_probe.py's cam1000: 256 problems x (16 positions x 4 headings of 90 degrees), m = 1
Each workload's coverable total T_q is the total of a quota call with quota = UINT64_MAX; the quotas are
ceil(p * T_q) for p = 0.5, 0.9 and 1.0.  Paths, all on the view call (cameras) or the m-fold call (the others):
  quota    the quota call, kmax = the group size
  (a) full the fixed-k call with k = the group size, today's way to a full cover; the answer is the prefix of its picks
  (b) known the fixed-k call with k = the quota call's largest npicked, as if the answer were known in advance
  (c) doubling  k = 8, 16, 32, .. until every problem's summed gain reaches its quota or its greedy stops, reading
           npicked and gain back after each try, as a careful caller would
Every path's pick, gain and npicked, cut at the first pick that reaches the quota, must equal the quota call's, and its
count must equal the quota call's where the path made exactly that many picks.  Times are CUDA events on the context's
stream after warm-up: median, min and max over the repeats.  `rounds` is the largest npicked, and `per_round_us` the
time a round adds, (t(rounds) - t(1)) / (rounds - 1) from the event times of the quota call and of (b) against the
same call with kmax = 1 and k = 1 (the loops run up to 65 536 rounds, too many kernel records for a profiler run).
`enqueue_ms` is the host time to enqueue one call with kmax = 1 (the quota call builds, launches and destroys its graph
in it), against the fixed-k call with k = 1; the difference is what capturing and instantiating the graph costs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from merge_probe import free_sources, gpu_info, shipped_map, timed  # noqa: E402
from window_probe import obstacle_map  # noqa: E402

U64_MAX = np.iinfo(np.uint64).max


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import visibility_heuristic_path_planner_b200 as vhp
    if not torch.cuda.is_available():
        raise SystemExit("cover_quota_probe needs a CUDA device")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g = np.random.default_rng(19)
    res = dict(probe="cover_quota", gpu=gpu_info(), workloads={})
    ctx = vhp.torch_context(0, stream)
    T = lambda fn: timed(torch, stream, fn, args.reps, args.warm)  # noqa: E731
    thr = 0.5
    occ16 = obstacle_map(vhp, torch, dev, 16384, 16384)
    occ1 = torch.from_numpy(shipped_map(g)[None]).to(dev)

    def cameras(occ_t, nprob, npos, nhead, R):
        xy = np.repeat(free_sources(g, occ_t.cpu().numpy(), nprob * npos), nhead, axis=0)
        heads = np.tile(np.arange(nhead) * (360.0 / nhead), nprob * npos)
        return xy, vhp.sensor_views(heads, 90, R)

    def workloads():
        xy = free_sources(g, occ16.cpu().numpy(), 65536)
        yield "g16384_m1", occ16, xy, None, 1, 32, 1
        yield "g16384_m2", occ16, xy, None, 1, 32, 2
        yield ("cam16384", occ16, *cameras(occ16, 1, 8192, 8, 32), 1, 32, 1)
        yield "c1000", occ1, free_sources(g, occ1.cpu().numpy(), 256 * 64), None, 256, 64, 1
        yield ("cam1000", occ1, *cameras(occ1, 256, 16, 4, 64), 256, 64, 1)

    all_equal = True
    for name, occ_t, xy, views, nprob, R, m in workloads():
        _, ny, nx = occ_t.shape
        n = xy.shape[0]
        K = n // nprob
        with torch.cuda.stream(stream):
            xy_t = torch.from_numpy(xy).to(dev)
            v_t = None if views is None else torch.from_numpy(views).to(dev)
            ptr_t = torch.arange(0, n + 1, K, dtype=torch.int64, device=dev)

            def outs(k):
                return [torch.empty((nprob, k), dtype=torch.int32, device=dev),
                        torch.empty((nprob, k), dtype=torch.int64, device=dev),
                        torch.empty((nprob,), dtype=torch.int32, device=dev),
                        torch.empty((nprob, ny, nx), dtype=torch.uint8, device=dev)]
            qo = outs(K) + [torch.empty((nprob,), dtype=torch.int64, device=dev)]
        stream.synchronize()
        ctx.prepare_maps_dev(occ_t)

        def quota_call(q_t, kmax, o):
            ctx.visibility_cover_quota_batch_dev(occ_t, xy_t, ptr_t, q_t, kmax, thr, R, vhp.RANGE_DISK, m=m,
                                                 pick_t=o[0], gain_t=o[1], npicked_t=o[2], count_t=o[3],
                                                 total_t=o[4] if len(o) > 4 else None, views_t=v_t)

        def fixed_call(k, o):
            if v_t is None:
                ctx.visibility_cover_greedy_mfold_batch_dev(occ_t, xy_t, ptr_t, k, m, thr, R, vhp.RANGE_DISK,
                                                            pick_t=o[0], gain_t=o[1], npicked_t=o[2], count_t=o[3])
            else:
                ctx.visibility_cover_greedy_view_batch_dev(occ_t, xy_t, v_t, ptr_t, k, m, thr, R, vhp.RANGE_DISK,
                                                           pick_t=o[0], gain_t=o[1], npicked_t=o[2], count_t=o[3])

        with torch.cuda.stream(stream):
            qmax = torch.full((nprob,), -1, dtype=torch.int64, device=dev)
            quota_call(qmax, K, qo)
            e1 = outs(1) + [torch.empty((nprob,), dtype=torch.int64, device=dev)]
        ctx.synchronize()
        one_round = dict(quota=T(lambda: quota_call(qmax, 1, e1)), fixed=T(lambda: fixed_call(1, e1)))
        coverable = qo[4].cpu().numpy().view(np.uint64).copy()
        w = dict(problems=nprob, candidates_per_problem=K, nx=nx, ny=ny, radius=R, shape="disk", threshold=thr, m=m,
                 views="90 degree cameras" if views is not None else None,
                 coverable_total=int(coverable.sum()), full_cover_npicked_max=int(qo[2].max().item()), fractions={})
        for p in (0.5, 0.9, 1.0):
            quota = np.ceil(p * coverable.astype(np.float64)).astype(np.uint64)
            quota = np.minimum(quota, coverable)  # p = 1.0: exactly the coverable total
            with torch.cuda.stream(stream):
                q_t = torch.from_numpy(quota.view(np.int64)).to(dev)
                quota_call(q_t, K, qo)
            ctx.synchronize()
            want = [x.cpu().numpy() for x in qo]
            kb = int(want[2].max())
            with torch.cuda.stream(stream):
                ob, oa = outs(max(kb, 1)), outs(K)
            d = dict(rounds=kb, npicked_total=int(want[2].sum()), paths={}, equal={})

            def doubling():
                k = 8
                while True:
                    with torch.cuda.stream(stream):
                        o = outs(k)
                    fixed_call(k, o)
                    ctx.synchronize()
                    npk, gain = o[2].cpu().numpy(), o[1].cpu().numpy().view(np.uint64)
                    done = (gain.sum(1, dtype=np.uint64) >= quota) | (npk < k) | (k >= K)
                    if done.all():
                        return o, k
                    k = min(2 * k, K)

            d["paths"]["quota"] = T(lambda: quota_call(q_t, K, qo))
            d["paths"]["a_full"] = T(lambda: fixed_call(K, oa))
            d["paths"]["b_known"] = T(lambda: fixed_call(kb, ob))
            d["paths"]["c_doubling"] = T(lambda: doubling())
            with torch.cuda.stream(stream):
                oc, kc = doubling()
            d["c_final_k"] = kc
            for path, o in (("a_full", oa), ("b_known", ob), ("c_doubling", oc)):
                if path == "a_full":
                    fixed_call(K, oa)
                elif path == "b_known":
                    fixed_call(kb, ob)
                ctx.synchronize()
                pk, gn, npk, cnt = (x.cpu().numpy() for x in o)
                ok = True
                for q in range(nprob):
                    j = int(want[2][q])
                    sums = np.concatenate([[0], np.cumsum(gn[q][:npk[q]].view(np.uint64).astype(object))])
                    jj = next((i for i, s in enumerate(sums) if s >= int(quota[q])), int(npk[q]))
                    ok &= jj == j and np.array_equal(pk[q][:j], want[0][q][:j]) and \
                        np.array_equal(gn[q][:j], want[1][q][:j])
                    if int(npk[q]) == j:
                        ok &= np.array_equal(cnt[q], want[3][q])
                d["equal"][path] = bool(ok)
                all_equal &= bool(ok)
            if kb > 1:
                d["per_round_us"] = dict(
                    quota=1e3 * (d["paths"]["quota"]["ms_median"] - one_round["quota"]["ms_median"]) / (kb - 1),
                    b_known=1e3 * (d["paths"]["b_known"]["ms_median"] - one_round["fixed"]["ms_median"]) / (kb - 1))
            d["quota_over_b"] = d["paths"]["quota"]["ms_median"] / d["paths"]["b_known"]["ms_median"]
            print(name, f"p={p}", json.dumps(d), flush=True)
            w["fractions"][str(p)] = d
            del ob, oa
        # host time to enqueue one call of one round: the quota call builds its graph in it
        w["one_round_ms"] = one_round
        eq, ef = [], []
        for _ in range(args.warm + args.reps):
            ctx.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                quota_call(qmax, 1, e1)
            eq.append((time.perf_counter() - t0) * 1e3)
            ctx.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                fixed_call(1, e1)
            ef.append((time.perf_counter() - t0) * 1e3)
        ctx.synchronize()
        eq, ef = eq[args.warm:], ef[args.warm:]
        w["enqueue_ms"] = dict(quota_median=float(np.median(eq)), fixed_median=float(np.median(ef)),
                               graph_build_ms=float(np.median(eq) - np.median(ef)))
        res["workloads"][name] = w
        del qo, e1
        torch.cuda.empty_cache()
    ctx.close()
    res["all_paths_equal"] = bool(all_equal)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
