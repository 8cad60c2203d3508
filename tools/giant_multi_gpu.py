#!/usr/bin/env python
"""Strip-partitioned planner on N GPUs (one rank per GPU, NCCL inside the library): every rank
checks its rows against the single-GPU planner it runs itself, rank 0 prints timings.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port 29533 tools/giant_multi_gpu.py [--size 2048] [--queries 3] [--spr 1]

BASELINE configs[4] shape: --size 8192 (dense random obstacles, multi-source planner).
--map mirrored: the same obstacles on one quarter, mirrored about the middle row and the middle column (an odd
side), every query from the centre to a point on one of the two axes: cells mirrored about the start tie on h, so
the first pushed of them has to win across ranks.  On two ranks of one strip each the middle row is rank 0's last.
torch.distributed (gloo) only carries the 128-byte NCCL id and the verdicts."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def giant_map(n, seed=8192):
    g = np.random.default_rng(seed)
    occ = np.ones((n, n), dtype=np.uint8)
    for _ in range(int(6000 * (n / 8192) ** 2)):
        x, y = int(g.integers(1, n)), int(g.integers(1, n))
        w, h = int(g.integers(8, 65)), int(g.integers(8, 65))
        occ[y:y + h, x:x + w] = 0
    return occ, g


def mirrored_map(n, queries):
    """(occ, queries): giant_map's obstacles on a quarter, mirrored about both axes of a (2m+1)^2 map, m = n // 2;
    start at the centre, ends on the axes"""
    m = n // 2
    q, g = giant_map(m + 1)
    occ = np.concatenate([q, q[:, -2::-1]], axis=1)
    occ = np.concatenate([occ, occ[-2::-1]], axis=0)
    out = []
    for k in range(queries):
        d = int(g.integers(m // 4, m))
        end = ((m, m + d), (m + d, m), (m, m - d), (m - d, m))[k % 4]
        out.append(((m, m), end))
        for x, y in ((m, m), end):
            occ[y, x] = occ[y, 2 * m - x] = occ[2 * m - y, x] = occ[2 * m - y, 2 * m - x] = 1
    assert np.array_equal(occ, occ[::-1]) and np.array_equal(occ, occ[:, ::-1])
    return occ, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--queries", type=int, default=3)
    ap.add_argument("--thr", type=float, default=0.3)
    ap.add_argument("--max-iter", type=int, default=60)
    ap.add_argument("--spr", type=int, default=1, help="strips per rank")
    ap.add_argument("--batch", type=int, default=0, help="iterations per snapshot (0: default)")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--map", choices=("random", "mirrored"), default="random")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    import visibility_heuristic_path_planner_b200 as vhp
    from visibility_heuristic_path_planner_b200.giant import GiantPlanner
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("gloo")
    if args.map == "mirrored":
        occ, queries = mirrored_map(args.size, args.queries)
    else:
        occ, g = giant_map(args.size)
        free = np.argwhere(occ != 0)
        picks = free[g.integers(0, len(free), 2 * args.queries)]
        queries = [((int(a[1]), int(a[0])), (int(b[1]), int(b[0]))) for a, b in zip(picks[::2], picks[1::2])]
    n = occ.shape[0]
    if world > 1:
        gp = GiantPlanner.from_torch_dist(occ, local, dist, strips_per_rank=args.spr)
    else:
        gp = GiantPlanner(occ, device=local, strips_per_rank=args.spr)
    if args.batch:
        gp.set_loop_mode(0, args.batch)
    ref_ctx = None if args.no_check else vhp.Context(local)
    out, all_same = [], True
    for qi, (start, end) in enumerate(queries):
        for rep in range(2):  # the second call is the timed one (graph / communicators warm)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            r = gp.solve(start, end, args.thr, args.max_iter, fields=(rep == 0 and not args.no_check))
            dt = time.perf_counter() - t0
            if rep == 0:
                first = r
        st = r["stats"]
        rec = dict(start=start, end=end, status=r["status"], nb=r["nb_of_sources"], iterations=st["iterations"],
                   path_length=r["path_length"], ms=dt * 1e3, loop_ms=st["loop_ms"],
                   ms_per_iteration=st["loop_ms"] / max(1, st["iterations"]), nccl_ms=st["nccl_ms"],
                   nccl_ops=st["nccl_ops"], halo_bytes_sent=st["halo_bytes_sent"], loop_mode=st["loop_mode"],
                   peer_handover=st["peer_handover"])
        if ref_ctx is not None:
            t0 = time.perf_counter()
            ref = ref_ctx.planner_batch(occ, [start + end], threshold=args.thr, max_iter=args.max_iter)
            rec["single_gpu_ms"] = (time.perf_counter() - t0) * 1e3
            nb = int(ref["nb_sources"][0])
            y0, y1 = first["rows"]
            same = (int(ref["status"][0]) == r["status"] and nb == r["nb_of_sources"]
                    and np.array_equal(ref["light_sources"][0][: nb + 1], r["light_sources"])
                    and float(ref["path_len"][0]) == r["path_length"]
                    and np.array_equal(ref["path"][0][: int(ref["path_n"][0])], r["path"])
                    and np.array_equal(ref["vg"][0][y0:y1], first["vg"])
                    and np.array_equal(ref["vis"][0][y0:y1], first["vis"])
                    and np.array_equal(ref["came"][0][y0:y1], first["came"]))
            rec["equal_single_gpu"] = bool(same)
            all_same &= bool(same)
        out.append(rec)
    verdicts = [all_same]
    if world > 1:
        verdicts = [None] * world
        dist.all_gather_object(verdicts, all_same)
    if rank == 0:
        print(json.dumps(dict(n=n, world=world, strips_per_rank=args.spr, all_ranks_equal=all(verdicts),
                              queries=out)), flush=True)
    gp.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not all(verdicts):
        sys.exit(1)


if __name__ == "__main__":
    main()
