#!/usr/bin/env python
"""bench.py -- headline benchmark: batched visibility sweep on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c2|c2s|c4] [--dump-outputs DIR]

A "step" is one pass of the hot path (computeVisibility) over one batch of
synthetic (map, source) pairs:
  c2 (default, BASELINE.json configs[1]): one empty 1000x1000 grid, 4096 light
      sources per GPU; output fp64-computed visibility stored as fp32.
  c2s: the same grid and batch size with the shipped settings.config environment
      (15 rectangles of 100-200 cells) and free-cell sources: the penumbra regime.
  c4 (configs[3] shape): 1024 random 256x256 obstacle maps x 16 sources per GPU.
Weak scaling: every rank sweeps its own batch (independent pairs, no data-path
collective); `value` = cells swept by all ranks / max-over-ranks device time.

Prints ONE JSON line (rank 0).  Keys follow the driver contract plus `roofline`,
`cpu_baseline`, `e2e`, `clocks`, `gpu_launches`.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Gcells/s visibility sweep (1000² grid, batched sources)"
DUMP_BYTES = 60 * 10**6  # --dump-outputs budget: a full batch is 16 GB


# ----------------------------------------------------------------------------
def workload(name, rank, world=1, use_device=True):
    """Synthetic batch for one rank: (maps uint8 [nmaps,ny,nx], src_xy, src_map, desc)."""
    if name == "c2":
        from visibility_heuristic_path_planner_b200.sharding import shard_batch
        nx = ny = 1000
        n = 4096 * world  # global batch, cut into contiguous blocks of 4096 per rank
        maps = np.ones((1, ny, nx), dtype=np.uint8)
        g = np.random.default_rng(1234)
        src = np.stack([g.integers(0, nx, n), g.integers(0, ny, n)], axis=1).astype(np.int32)
        src[0] = (500, 500)  # the reference's benchmarkSeries case
        maps, src, _, _ = shard_batch(maps, src, None, rank, world)
        return maps, src, None, ("1000x1000 empty grid, 4096 light sources per GPU "
                                 "(global batch PCG64 seed 1234, contiguous block per rank)")
    if name == "c2s":
        # the headline grid with the shipped settings.config environment (15 rectangles of
        # 100-200 cells, config/settings.config:8-14): the DP (penumbra) regime at 1000x1000
        nx = ny = 1000
        n = 4096
        g = np.random.default_rng(2500 + rank)
        maps = np.ones((1, ny, nx), dtype=np.uint8)
        for _ in range(15):
            x, y = int(g.integers(1, nx)), int(g.integers(1, ny))
            w, h = int(g.integers(100, 201)), int(g.integers(100, 201))
            maps[0, y:y + h, x:x + w] = 0
        free = np.argwhere(maps[0] != 0)
        pick = free[g.integers(0, len(free), n)]
        src = np.ascontiguousarray(pick[:, ::-1]).astype(np.int32)
        return maps, src, None, ("1000x1000 grid with the shipped settings.config environment (15 rectangles "
                                 "100-200 cells, %.1f%% occupied), 4096 free-cell light sources per GPU"
                                 % (100.0 * (1.0 - maps.mean())))
    if name == "c2d":
        # the headline grid crowded with small obstacles (400 rectangles of 8-40 cells, the
        # C4 / C5 obstacle sizes): penumbra nearly everywhere, few lit or dark tiles
        nx = ny = 1000
        n = 4096
        g = np.random.default_rng(2600 + rank)
        maps = np.ones((1, ny, nx), dtype=np.uint8)
        for _ in range(400):
            x, y = int(g.integers(1, nx)), int(g.integers(1, ny))
            w, h = int(g.integers(8, 41)), int(g.integers(8, 41))
            maps[0, y:y + h, x:x + w] = 0
        free = np.argwhere(maps[0] != 0)
        pick = free[g.integers(0, len(free), n)]
        src = np.ascontiguousarray(pick[:, ::-1]).astype(np.int32)
        return maps, src, None, ("1000x1000 grid with 400 random rectangles of 8-40 cells (%.1f%% occupied), "
                                 "4096 free-cell light sources per GPU" % (100.0 * (1.0 - maps.mean())))
    if name == "c4":
        # BASELINE configs[3]: 16384 random 256 x 256 obstacle maps x 16 sources over 8 GPUs = 2048 maps
        # (32768 pairs) per GPU.  The maps are generated ON THE DEVICE where there is one
        # (vhp_environment_generate_batch_dev: the reference's rectangle rule, src/environment.cpp:57-79,
        # with counter-based draws; map index = global index of the map) and read back once to pick
        # 16 free source cells per map.
        nx = ny = 256
        nmaps, per = 2048, 16
        g = np.random.default_rng(4321 + rank)
        maps = None
        try:
            import torch
            if use_device and torch.cuda.is_available():
                import visibility_heuristic_path_planner_b200 as vhp
                dev_i = int(os.environ.get("LOCAL_RANK", "0"))
                c = vhp.Context(dev_i)
                t = torch.empty((nmaps, ny, nx), dtype=torch.uint8, device=torch.device("cuda", dev_i))
                c.generate_environments_dev(t, 12, 8, 40, 8, 40, seed=4321, first_map=rank * nmaps)
                c.synchronize()
                maps = t.cpu().numpy()
                c.close()
        except Exception:
            maps = None
        if maps is None:  # no GPU (the reference arm's config string only needs the shape)
            maps = np.ones((nmaps, ny, nx), dtype=np.uint8)
            for m in range(nmaps):
                for _ in range(12):
                    x, y = int(g.integers(1, nx)), int(g.integers(1, ny))
                    w, h = int(g.integers(8, 41)), int(g.integers(8, 41))
                    maps[m, y:y + h, x:x + w] = 0
        src = np.zeros((nmaps * per, 2), dtype=np.int32)
        smap = np.repeat(np.arange(nmaps, dtype=np.int32), per)
        flat = maps.reshape(nmaps, -1) != 0
        for m in range(nmaps):
            free = np.flatnonzero(flat[m])
            pick = free[g.integers(0, len(free), per)]
            src[m * per:(m + 1) * per, 0] = pick % nx
            src[m * per:(m + 1) * per, 1] = pick // nx
        return maps, src, smap, ("2048 random 256x256 maps (12 rectangles 8-40, generated on the device) x 16 "
                                 "free-cell sources per GPU")
    raise SystemExit(f"unknown workload {name}")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu), "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank on the CPUs of its GPU's NUMA node, so that the pinned host buffers of the
    end-to-end leg are allocated next to the GPU's PCIe root (ranks launched by torchrun are not
    bound; with several ranks the D2H streams otherwise cross the socket interconnect).
    Best effort: silently does nothing where sysfs does not expose the topology."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(gpu_index)
        if hasattr(pr, "pci_bus_id"):
            dev = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        else:
            bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i",
                                  str(gpu_index)], capture_output=True, text=True, timeout=20).stdout.strip()
            dom, rest = bus.split(":", 1)
            dev = f"{dom[-4:].lower()}:{rest.lower()}"
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash():
    """SHA-256 (first 16 hex digits) of the sources of the dominant kernel: ties an ncu capture to
    the code it was taken from."""
    import hashlib
    h = hashlib.sha256()
    for f in ("sweep_tile_body.cuh", "kernels_sweep_tile.cu", "sweep_common.cuh"):
        h.update(open(os.path.join(ROOT, "visibility_heuristic_path_planner_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(workload_name, pairs):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (per pair on a
    subset of the batch, scaled to this launch's pairs) -- only while the capture was taken from
    the kernel sources that are being benchmarked (tools/capture_traffic.py stamps their hash);
    otherwise null."""
    p = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(p):
        j = json.load(open(p))
        d = j.get(workload_name)
        if d and j.get("kernel_source_hash") == kernel_source_hash():
            return d["dram_bytes_per_pair"] * pairs
    return None


def dump_outputs(path, out_t):
    """--dump-outputs: the fields of a fixed sample of the batch's pairs (PCG64 seed 0, as many as
    DUMP_BYTES holds, in pair order) as DIR/visibility.npy [pairs, ny, nx], in the stored dtype, and
    their indices in the batch as DIR/visibility_pairs.npy (float64), so that two builds can be
    compared output for output."""
    import torch
    n = out_t.shape[0]
    k = max(1, min(n, DUMP_BYTES // (out_t[0].numel() * out_t.element_size())))
    idx = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "visibility.npy"), out_t[torch.from_numpy(idx).to(out_t.device)].cpu().numpy())
    np.save(os.path.join(path, "visibility_pairs.npy"), idx.astype(np.float64))


def bench_config(workload_name, desc, nx, ny, n, store, world):
    """The `config` object of the JSON line -- the same for both arms (--impl ours / reference)."""
    esz = 4 if store == "f32" else 8
    return {"workload": f"{workload_name}: {desc}", "grid": [nx, ny], "pairs_per_gpu": n, "store": store,
            "parallelism": f"batch-shard x{world}, no collective",
            "l2": "outputs (%.1f GB per step) exceed the 126 MB L2; the shared map is L2-resident by design"
                  % (n * nx * ny * esz / 1e9)}


# ----------------------------------------------------------------------------
def run_reference(args, rank, world):
    """--impl reference: the reference's own computeVisibility() on the host cores."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_py import Oracle, Ref
    maps, src, smap, desc = workload(args.workload, 0, max(1, args.gpus), use_device=False)  # (no GPU code in this arm)
    ny, nx = maps.shape[1:]
    cores = os.cpu_count() or 1
    per_step = min(len(src), 16 * cores)
    occ = maps[0].astype(np.float64)
    if Ref.available("fast"):
        ref, kind = Ref("fast"), "reference"
        flags = ref.flags()

        def step(lo):
            return ref.time_compute_visibility(occ, src[lo:lo + per_step], nthreads=cores)
    else:  # oracle port, single thread
        ora, kind, cores, flags = Oracle(), "port", 1, "-O2 -ffp-contract=off"
        per_step = min(per_step, 32)

        def step(lo):
            t0 = time.perf_counter()
            for sx, sy in src[lo:lo + per_step]:
                ora.compute_visibility(occ, sx, sy)
            return time.perf_counter() - t0
    for w in range(args.warmup):
        step(0)
    secs = [step((i * per_step) % max(1, len(src) - per_step + 1)) for i in range(args.steps)]
    t = sum(secs) / len(secs)
    val = per_step * nx * ny / t / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Gcells/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.workload, desc, nx, ny, len(src), args.store, max(1, args.gpus)),
            "cpu_baseline": {"value": val, "unit": "Gcells/s", "cores": cores, "kind": kind,
                             "sample": f"each step = {per_step} sources of the workload's batch (a bounded sample, the rate "
                                       f"is per cell), one solver instance per thread on {cores} threads, fp64 "
                                       f"Field<double> output, flags {flags}"},
            "e2e": {"value": val, "unit": "Gcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline(maps, src, nx, ny):
    """Reference CPU solver on this box's host cores (bounded sample)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_py import Oracle, Ref
    occ = maps[0].astype(np.float64)
    cores = os.cpu_count() or 1
    if Ref.available("fast"):
        ref = Ref("fast")
        n1 = min(len(src), 48)
        t1 = ref.time_compute_visibility(occ, src[:n1], nthreads=1)
        nall = min(len(src), 96 * cores)
        ref.time_compute_visibility(occ, src[:cores], nthreads=cores)  # warm-up
        tall = ref.time_compute_visibility(occ, src[:nall], nthreads=cores)
        return {"value": nall * nx * ny / tall / 1e9, "unit": "Gcells/s", "cores": cores,
                "kind": "reference",
                "value_1core": n1 * nx * ny / t1 / 1e9,
                "sample": (f"reference computeVisibility() ({ref.flags()}): {nall} sources on "
                           f"{cores} threads (one solver instance per thread); 1-core figure from {n1} sources")}
    ora = Oracle()
    n1 = min(len(src), 32)
    t0 = time.perf_counter()
    for sx, sy in src[:n1]:
        ora.compute_visibility(occ, sx, sy)
    t1 = time.perf_counter() - t0
    return {"value": n1 * nx * ny / t1 / 1e9, "unit": "Gcells/s", "cores": 1, "kind": "port",
            "sample": f"oracle/vhp_oracle.c (-O2 -ffp-contract=off), {n1} sources, 1 thread"}



def _timed_dev(stream, fn, reps, warm=3):
    """Average milliseconds of fn() enqueued on `stream` (CUDA events on that stream)."""
    import torch
    with torch.cuda.stream(stream):
        for _ in range(warm):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
    stream.synchronize()
    return e0.elapsed_time(e1) / reps


def _ref_fast():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_py import Ref
    return Ref("fast") if Ref.available("fast") else None


def c1_leg(vhp, ctx, stream, dev, local_rank, with_cpu):
    """BASELINE configs[0]: 101 x 101 random environment (parser.h defaults, seed 2), ONE light
    source, stand-alone visibility -- the reference's only published figure (README.md:9,
    "~55 kHz").  Latency of one sweep, not throughput."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_py import Oracle
    occ = (Oracle().generate_environment(101, 101, 10, 10, 20, 10, 20, 2) != 0).astype(np.uint8)[None]
    src = np.array([[5, 5]], np.int32)
    occ_t, src_t = torch.from_numpy(occ).to(dev), torch.from_numpy(src).to(dev)
    out_t = torch.empty((1, 101, 101), dtype=torch.float64, device=dev)
    ctx.prepare_maps_dev(occ_t)
    ms = _timed_dev(stream, lambda: ctx.visibility_batch_dev(occ_t, src_t, out_t), 2000, 20)
    # the same sweep 4096 times in one launch: what the kernel does when it is not a single CTA
    nb = 4096
    srcb = torch.from_numpy(np.repeat(src, nb, 0)).to(dev)
    outb = torch.empty((nb, 101, 101), dtype=torch.float64, device=dev)
    msb = _timed_dev(stream, lambda: ctx.visibility_batch_dev(occ_t, srcb, outb), 20)
    hctx = vhp.Context(local_rank)
    hctx.visibility_batch(occ, src, dtype=vhp.F64)
    t0 = time.perf_counter()
    for _ in range(200):
        hctx.visibility_batch(occ, src, dtype=vhp.F64)
    host_us = (time.perf_counter() - t0) / 200 * 1e6
    hctx.close()
    out = {"workload": "101x101 random environment (10 rectangles 10-20, glibc rand seed 2), one light source (5,5), fp64",
           "device_us_per_sweep": ms * 1e3, "device_khz": 1.0 / ms,
           "host_call_us_per_sweep": host_us, "host_call_khz": 1e3 / host_us,
           "batched_us_per_sweep": msb * 1e3 / nb, "batched_khz": nb / msb,
           "note": "device = vhp_visibility_batch_dev with one pair, maps prepared, back-to-back launches timed with "
                   "CUDA events; host_call = vhp_visibility_batch (upload, pack, sweep, 82 KB back, synchronous); "
                   "batched = 4096 pairs per launch / time",
           "published": {"value_khz": 55.0, "hardware": "i9-13980HX, one core", "source": "README.md:9"}}
    ref = _ref_fast() if with_cpu else None
    if ref is not None:
        t = ref.time_compute_visibility(occ[0].astype(np.float64), np.repeat(src, 2000, 0), nthreads=1)
        out["cpu_reference"] = {"us_per_sweep": t / 2000 * 1e6, "khz": 2000 / t / 1e3, "cores": 1, "kind": "reference",
                                "sample": f"reference computeVisibility() ({ref.flags()}), 2000 repetitions, one thread"}
    return out


def c3_leg(vhp, local_rank, with_cpu):
    """BASELINE configs[2]: images/maze_5.png (242 x 322), start {118,317}, end {123,10} (bottom-left
    origin), threshold 0.2: 112 light sources, path length 1341.7118586874171 (SURVEY 8c).  The map
    comes from the committed golden fixture (the PNG is not on the GPU box)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "maze5.npz"))
    ny, nx = (int(v) for v in g["shape"])
    occ = np.unpackbits(g["occ_bits"])[: ny * nx].reshape(ny, nx).astype(np.uint8)
    start, end = tuple(int(v) for v in g["start"]), tuple(int(v) for v in g["end"])
    se1 = np.array([start + end], np.int32)
    ctx = vhp.Context(local_rank)
    out = {"workload": f"maze_5 ({nx}x{ny}), start {start} end {end} (internal frame), threshold 0.2, max_iter 250"}

    def timed(se, reps, **kw):
        r = ctx.planner_batch(occ, se, threshold=0.2, max_iter=250, fields=False, **kw)
        t0 = time.perf_counter()
        for _ in range(reps):
            r = ctx.planner_batch(occ, se, threshold=0.2, max_iter=250, fields=False, **kw)
        return (time.perf_counter() - t0) / reps, r

    t1, r = timed(se1, 5)
    assert int(r["status"][0]) == 0 and int(r["nb_sources"][0]) == 112, (r["status"], r["nb_sources"])
    assert float(r["path_len"][0]) == float(g["thr020_len"][0])
    out["single"] = {"ms_per_solve": t1 * 1e3, "solves_per_s": 1.0 / t1, "sources": 112,
                     "path_length": float(r["path_len"][0]),
                     "route": "one problem on the whole GPU: sweeps over many CTAs, loop as a CUDA-graph WHILE node"}
    for mode, name in ((3, "single_readback_per_iteration"),):
        ctx.set_planner_loop(mode)
        t, r2 = timed(se1, 5)
        assert float(r2["path_len"][0]) == float(r["path_len"][0])
        out[name] = {"ms_per_solve": t * 1e3}
    ctx.set_planner_loop(0)
    ctx.set_grid_sweep(0)  # the persistent one-CTA-per-problem kernel
    t, r2 = timed(se1, 3)
    assert float(r2["path_len"][0]) == float(r["path_len"][0])
    out["single_one_cta"] = {"ms_per_solve": t * 1e3}
    ctx.set_grid_sweep(1)
    nb = 1024
    tb, rb = timed(np.repeat(se1, nb, 0), 2)
    assert (rb["nb_sources"] == 112).all() and (rb["path_len"] == r["path_len"][0]).all()
    out["batch_identical"] = {"problems": nb, "ms_per_batch": tb * 1e3, "solves_per_s": nb / tb}
    rng = np.random.default_rng(5)
    free = np.argwhere(occ != 0)
    a, b = free[rng.integers(0, len(free), nb)], free[rng.integers(0, len(free), nb)]
    sed = np.stack([a[:, 1], a[:, 0], b[:, 1], b[:, 0]], 1).astype(np.int32)
    td, rd = timed(sed, 2)
    out["batch_distinct"] = {"problems": nb, "ms_per_batch": td * 1e3, "solves_per_s": nb / td,
                             "solved": int((rd["status"] == 0).sum()), "max_iter_hit": int((rd["status"] == 5).sum()),
                             "mean_sources": float(rd["nb_sources"].mean())}
    ctx.close()
    ref = _ref_fast() if with_cpu else None
    if ref is not None:
        cores = os.cpu_count() or 1
        s1, _ = ref.time_solve(occ.astype(np.float64), se1, 0.2, 250, nthreads=1)
        sn, _ = ref.time_solve(occ.astype(np.float64), np.repeat(se1, cores, 0), 0.2, 250, nthreads=cores)
        out["cpu_reference"] = {"ms_per_solve_1core": s1 * 1e3, "solves_per_s_1core": 1.0 / s1,
                                "solves_per_s_all_cores": cores / sn, "cores": cores, "kind": "reference",
                                "sample": f"reference solve() ({ref.flags()}): one solve on one thread; {cores} copies "
                                          f"of it on {cores} threads"}
    return out


def raycast_leg(vhp, ctx, stream, dev, with_cpu):
    """BASELINE configs[1] second half, "sweep vs raycasting" (README.md:13, benchmark() :226-235):
    the all-targets ray casting loop on the empty 1000 x 1000 grid for a 64-source subset of the
    batch, beside the sweep of the same 64 sources."""
    import torch
    maps, src, _, _ = workload("c2", 0, 1)
    src = np.ascontiguousarray(src[:64])
    ny, nx = maps.shape[1:]
    occ_t, src_t = torch.from_numpy(maps).to(dev), torch.from_numpy(src).to(dev)
    out_t = torch.empty((64, ny, nx), dtype=torch.float32, device=dev)
    ctx.prepare_maps_dev(occ_t)
    ms_ray = _timed_dev(stream, lambda: ctx.raycast_batch_dev(occ_t, src_t, out_t), 3, 1)
    ms_swp = _timed_dev(stream, lambda: ctx.visibility_batch_dev(occ_t, src_t, out_t), 20, 3)
    rays = 64 * nx * ny
    # cell visits of the Bresenham walks: max(|dx|, |dy|) per ray
    xs, ys = np.arange(nx), np.arange(ny)
    visits = sum(int(np.maximum(np.abs(xs[None, :] - sx), np.abs(ys[:, None] - sy)).sum()) for sx, sy in src)
    out = {"workload": "empty 1000x1000 grid, 64 light sources (the first 64 of the c2 batch), every cell a target",
           "raycast_ms": ms_ray, "rays_per_s": rays / ms_ray * 1e3, "cell_visits_per_s": visits / ms_ray * 1e3,
           "sweep_ms_same_sources": ms_swp, "sweep_vs_raycast": ms_ray / ms_swp,
           "note": "sweep_vs_raycast = ray-casting time / sweep time for the same 64 sources on the GPU (64 pairs "
                   "do not fill the machine for either kernel); the reference reports this ratio for one source on "
                   "one core (README.md:13: ~80x; Samples/benchmark_results.txt N=971: 135x)"}
    ref = _ref_fast() if with_cpu else None
    if ref is not None:
        occ = maps[0].astype(np.float64)
        t0 = time.perf_counter()
        ref.raycast_all(occ, int(src[0][0]), int(src[0][1]))
        t_ray = time.perf_counter() - t0
        t_swp = ref.time_compute_visibility(occ, src[:8], nthreads=1) / 8
        out["cpu_reference"] = {"raycast_ms_per_source": t_ray * 1e3, "sweep_ms_per_source": t_swp * 1e3,
                                "ratio": t_ray / t_swp, "cores": 1, "kind": "reference",
                                "sample": f"reference raycasting loop for one source and computeVisibility() for 8 "
                                          f"({ref.flags()}), one thread"}
    return out

def planner_workload(rank):
    """Batched planner problems: 64 random 256x256 obstacle maps x 128 (start, end) pairs."""
    nx = ny = 256
    nmaps, per = 64, 128
    g = np.random.default_rng(777 + rank)
    maps = np.ones((nmaps, ny, nx), dtype=np.uint8)
    for m in range(nmaps):
        for _ in range(12):
            x, y = int(g.integers(1, nx)), int(g.integers(1, ny))
            w, h = int(g.integers(8, 41)), int(g.integers(8, 41))
            maps[m, y:y + h, x:x + w] = 0
    se = np.zeros((nmaps * per, 4), dtype=np.int32)
    pmap = np.repeat(np.arange(nmaps, dtype=np.int32), per)
    for m in range(nmaps):
        free = np.argwhere(maps[m] != 0)
        a = free[g.integers(0, len(free), per)]
        b = free[g.integers(0, len(free), per)]
        se[m * per:(m + 1) * per] = np.stack([a[:, 1], a[:, 0], b[:, 1], b[:, 0]], axis=1)
    return maps, se, pmap


def executed_sweeps(r):
    """Sweeps the planner really ran per problem: nb_of_sources, except that a problem stuck on a
    fixed point (the same source selected again, SURVEY A.2 item 7) stops sweeping there while the
    reference's list is filled up to max_iter."""
    ls, nb = r["light_sources"], r["nb_sources"]
    same = (ls[:, 1:] == ls[:, :-1]).all(axis=2)          # ls[i] == ls[i-1], i = 1..
    idx = np.arange(1, ls.shape[1])[None, :]
    same &= (idx <= nb[:, None]) & (r["status"][:, None] == 5)
    first = np.where(same.any(axis=1), same.argmax(axis=1) + 1, nb)
    return np.minimum(first, nb)


def planner_leg(vhp, local_rank, rank, world, dist, dev, with_cpu):
    """Secondary metric of BASELINE.json: planner solves/s (solve() + reconstructPath() per
    problem, whole loop on the device), through the host-buffer C-ABI call, plus the device-
    resident rate of the same batch and its roofline (SURVEY 8d: 29 B per cell and iteration)."""
    import torch
    maps, se, pmap = planner_workload(rank)
    thr, max_iter = 0.5, 100
    nmaps, ny, nx = maps.shape
    ctx = vhp.Context(local_rank)
    ctx.planner_batch(maps, se, prob_map=pmap, threshold=thr, max_iter=max_iter, fields=False)  # warm-up
    torch.cuda.synchronize()
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        r = ctx.planner_batch(maps, se, prob_map=pmap, threshold=thr, max_iter=max_iter, fields=False)
    torch.cuda.synchronize()
    t = (time.perf_counter() - t0) / reps
    ctx.close()
    # device-resident: inputs and small outputs stay on the GPU, CUDA events on the launch stream
    stream = torch.cuda.Stream(dev)
    dctx = vhp.torch_context(local_rank, stream)
    cap = max_iter + 2
    n = len(se)
    occ_t, se_t, pm_t = (torch.from_numpy(a).to(dev) for a in (maps, se, pmap))
    o = dict(status=torch.zeros(n, dtype=torch.int32, device=dev), nb=torch.zeros(n, dtype=torch.int32, device=dev),
             ls=torch.zeros((n, cap, 2), dtype=torch.int32, device=dev), plen=torch.zeros(n, dtype=torch.float64, device=dev),
             pn=torch.zeros(n, dtype=torch.int32, device=dev), path=torch.zeros((n, cap, 2), dtype=torch.int32, device=dev))
    po = vhp.PlannerOut(o["status"].data_ptr(), o["nb"].data_ptr(), o["ls"].data_ptr(), o["plen"].data_ptr(),
                        o["pn"].data_ptr(), o["path"].data_ptr(), None, None, None)
    import ctypes as C
    dctx.prepare_maps_dev(occ_t)

    def dev_step():
        st = dctx.lib.vhp_planner_batch_dev(dctx.h, occ_t.data_ptr(), nmaps, nx, ny, se_t.data_ptr(), pm_t.data_ptr(),
                                            n, thr, max_iter, cap, vhp.F64, C.byref(po))
        assert st == 0, dctx.lib.vhp_last_error(dctx.h)
    ms_dev = _timed_dev(stream, dev_step, 3, 1)
    assert np.array_equal(o["nb"].cpu().numpy(), r["nb_sources"]) and np.array_equal(o["plen"].cpu().numpy(), r["path_len"])
    dctx.close()
    if world > 1:
        tt = torch.tensor([t, ms_dev], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t, ms_dev = float(tt[0].item()), float(tt[1].item())
    sweeps = int(executed_sweeps(r).sum())
    peak, _ = measured_peak()
    alg = 29.0 * nx * ny * sweeps  # occ 1 + vis 8 W + vg 8 R + 8 W + parent 4 R (fp64 working set), SURVEY 8d
    out = {"metric": "planner solves/s", "value": world * n / t, "unit": "solves/s",
           "problems_per_gpu": n, "ms_per_batch": t * 1e3,
           "workload": "64 random 256x256 maps (12 rectangles 8-40) x 128 (start,end) pairs per GPU, "
                       "threshold 0.5, max_iter 100; host-buffer vhp_planner_batch, small outputs only",
           "solved": int((r["status"] == 0).sum()), "max_iter_hit": int((r["status"] == 5).sum()),
           "mean_sources": float(r["nb_sources"].mean()), "light_sources": int(r["nb_sources"].sum()),
           "sweeps": sweeps,
           "device": {"ms_per_batch": ms_dev, "solves_per_s": world * n / ms_dev * 1e3,
                      "api": "vhp_planner_batch_dev, maps prepared, inputs and outputs resident, CUDA events"},
           "roofline": {"bound": "hbm", "achieved": alg / ms_dev / 1e6, "peak": peak, "unit": "GB/s",
                        "frac": alg / ms_dev / 1e6 / peak, "traffic": None, "kernel": "planner_kernel",
                        "algorithmic_bytes_per_launch": alg,
                        "note": "29 B per cell and executed sweep (SURVEY 8d) x %d sweeps of 256x256 cells; "
                                "device-resident batch time" % sweeps}}
    if with_cpu and rank == 0:
        ref = _ref_fast()
        if ref is not None:
            cores = os.cpu_count() or 1
            nm = 2  # bounded sample: 2 of the 64 maps
            secs = 0.0
            for m in range(nm):
                sel = se[pmap == m]
                secs += ref.time_solve(maps[m].astype(np.float64), sel, thr, max_iter, nthreads=cores)[0]
            n_cpu = int((pmap < nm).sum())
            out["cpu_reference"] = {"value": n_cpu / secs, "unit": "solves/s", "cores": cores,
                                    "kind": "reference",
                                    "sample": f"reference solve() ({ref.flags()}), {n_cpu} problems of the "
                                              f"same batch on {cores} threads"}
    return out


def giant_map(n=8192, seed=8192):
    g = np.random.default_rng(seed)
    occ = np.ones((n, n), dtype=np.uint8)
    for _ in range(int(6000 * (n / 8192) ** 2)):
        x, y = int(g.integers(1, n)), int(g.integers(1, n))
        w, h = int(g.integers(8, 65)), int(g.integers(8, 65))
        occ[y:y + h, x:x + w] = 0
    return occ, g


def giant_leg(vhp, local_rank, rank, world, dist, check=True, size=8192, queries=4):
    """BASELINE configs[4]: ONE dense random-obstacle 8192 x 8192 map, multi-source planner, the
    rows partitioned into one strip per GPU (NCCL halo rows + arg-min key exchange inside the
    library, vhp_giant_*).  On one GPU the same engine runs with a single strip.  With several
    ranks every rank compares its rows of the first query's fields, and every query's light
    sources and path, with the single-GPU planner it runs itself."""
    from visibility_heuristic_path_planner_b200.giant import GiantPlanner
    occ, g = giant_map(size)
    free = np.argwhere(occ != 0)
    picks = free[g.integers(0, len(free), 2 * queries)]
    qs = [((int(a[1]), int(a[0])), (int(b[1]), int(b[0]))) for a, b in zip(picks[::2], picks[1::2])]
    thr, max_iter = 0.3, 60
    if world > 1:
        gp = GiantPlanner.from_torch_dist(occ, local_rank, dist)
    else:
        gp = GiantPlanner(occ, device=local_rank)
    gp.solve(qs[0][0], qs[0][1], thr, max_iter, fields=False)  # warm-up: graph / communicators
    recs, firsts = [], None
    for qi, (a, b) in enumerate(qs):
        if world > 1:
            dist.barrier()
        r = gp.solve(a, b, thr, max_iter, fields=(check and qi == 0 and world > 1))
        if qi == 0:
            firsts = r
        st = r["stats"]
        recs.append(dict(status=r["status"], sources=r["nb_of_sources"], iterations=st["iterations"],
                         path_length=r["path_length"], loop_ms=st["loop_ms"], solve_ms=st["solve_ms"],
                         nccl_ms=st["nccl_ms"], halo_bytes_sent=st["halo_bytes_sent"], ls=r["light_sources"],
                         path=r["path"]))
    equal = None
    if check and world > 1:
        ctx = vhp.Context(local_rank)
        same = True
        for qi, ((a, b), rec) in enumerate(zip(qs, recs)):
            ref = ctx.planner_batch(occ, [a + b], threshold=thr, max_iter=max_iter, fields=(qi == 0))
            nb = int(ref["nb_sources"][0])
            same &= (int(ref["status"][0]) == rec["status"] and nb == rec["sources"]
                     and np.array_equal(ref["light_sources"][0][: nb + 1], rec["ls"])
                     and float(ref["path_len"][0]) == rec["path_length"]
                     and np.array_equal(ref["path"][0][: int(ref["path_n"][0])], rec["path"]))
            if qi == 0:
                y0, y1 = firsts["rows"]
                same &= (np.array_equal(ref["vg"][0][y0:y1], firsts["vg"])
                         and np.array_equal(ref["vis"][0][y0:y1], firsts["vis"])
                         and np.array_equal(ref["came"][0][y0:y1], firsts["came"]))
        ctx.close()
        verdicts = [None] * world
        dist.all_gather_object(verdicts, bool(same))
        equal = all(verdicts)
    loop_mode = gp.solve(qs[0][0], qs[0][1], thr, 1, fields=False)["stats"]["loop_mode"]
    gp.close()
    its = sum(q["iterations"] for q in recs)
    loop = sum(q["loop_ms"] for q in recs)
    nccl = sum(q["nccl_ms"] for q in recs)
    return {"workload": f"one dense random-obstacle {size}x{size} map ({int(6000 * (size / 8192) ** 2)} rectangles 8-64, "
                        f"{100.0 * (1.0 - occ.mean()):.1f}% occupied), {queries} (start, end) queries, threshold {thr}, "
                        f"max_iter {max_iter}; fp64 working fields; {world} strip(s), one per GPU",
            "ranks": world, "queries": queries, "iterations": its, "ms_per_iteration": loop / max(1, its),
            "ms_per_query": loop / queries,
            "solve_ms_per_query_host_wall": sum(q["solve_ms"] for q in recs) / queries,
            "halo_bytes_sent_per_iteration_rank0": (sum(q["halo_bytes_sent"] for q in recs) / max(1, its)),
            "nccl_time_share_rank0": (nccl / loop) if loop > 0 and world > 1 else 0.0,
            "nccl_note": "device time between events around rank 0's NCCL calls (ncclSend / ncclRecv of the halo rows, "
                         "ncclAllGather of the 32-byte key) / loop time; it includes waiting for the neighbour's strip",
            "loop": {1: "CUDA-graph WHILE node", 2: "batches of 4 iterations, snapshot one batch behind",
                     3: "read-back per iteration"}.get(loop_mode, loop_mode),
            "equal_single_gpu": equal,
            "per_query": [dict(sources=q["sources"], iterations=q["iterations"], status=q["status"],
                               path_length=q["path_length"], loop_ms=q["loop_ms"]) for q in recs]}


# ----------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c2s", "c2d", "c4"])
    ap.add_argument("--store", default="f32", choices=["f32", "f64"])
    ap.add_argument("--pairs", type=int, default=0, help="override pairs per GPU (profiling only)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-planner", action="store_true")
    ap.add_argument("--no-penumbra", action="store_true")
    ap.add_argument("--no-giant", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the C1 / C3 / ray-casting legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the fields of the last timed step to DIR/visibility.npy "
                         "and their pair indices to DIR/visibility_pairs.npy (rank 0's batch only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import visibility_heuristic_path_planner_b200 as vhp

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    # stdout carries the JSON line only: whatever libraries print (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    maps, src, smap, desc = workload(args.workload, rank, world)
    if args.pairs:
        src = np.ascontiguousarray(src[:args.pairs])
        smap = None if smap is None else np.ascontiguousarray(smap[:args.pairs])
        desc += f" [first {len(src)} pairs only]"
    nmaps, ny, nx = maps.shape
    n = len(src)
    cells = n * nx * ny
    tdt = torch.float32 if args.store == "f32" else torch.float64
    esz = 4 if args.store == "f32" else 8

    stream = torch.cuda.Stream(dev)
    ctx = vhp.torch_context(local_rank, stream)
    occ_t = torch.from_numpy(maps).to(dev)
    src_t = torch.from_numpy(src).to(dev)
    smap_t = None if smap is None else torch.from_numpy(smap).to(dev)
    out_t = torch.empty((n, ny, nx), dtype=tdt, device=dev)
    # inputs resident in HBM when the timed region starts: the maps and their bit planes (the
    # kernel's input layout, packed once per batch of maps)
    with torch.cuda.stream(stream):
        ctx.prepare_maps_dev(occ_t)
    torch.cuda.synchronize()

    def step():
        ctx.visibility_batch_dev(occ_t, src_t, out_t, smap_t)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
        if args.dump_outputs:
            out_t.fill_(float("nan"))  # what is dumped must come from the timed steps
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launches
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    with torch.cuda.stream(stream):
        evs[0].record(stream)
        for i in range(args.steps):
            step()
            evs[i + 1].record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launches - launches0
    ctx.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_t)
    total_ms = evs[0].elapsed_time(evs[-1])
    step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms_max = float(t.item())
    else:
        total_ms_max = total_ms
    ms_per_step = total_ms_max / args.steps
    value = cells * world / (ms_per_step * 1e-3) / 1e9

    # quick result sanity (not timed): the batch was really computed
    chk = out_t[0].double().sum().item()
    if args.workload == "c2":  # empty grid: everything lit except the never-written borders
        sx0, sy0 = int(src[0][0]), int(src[0][1])
        expect = nx * ny - (ny if sx0 > 0 else 0) - (nx if sy0 > 0 else 0) + (1 if sx0 > 0 and sy0 > 0 else 0)
        assert chk == expect, (chk, expect)

    # ---- end-to-end through the host-buffer C-ABI entry point ------------------
    e2e = None
    if not args.no_e2e:
        # host threads of the packed result transport: share the cores between the ranks of a box
        if world > 1 and "VHP_HOST_THREADS" not in os.environ:
            os.environ["VHP_HOST_THREADS"] = str(max(1, (os.cpu_count() or 1) // world))
        host_ctx = vhp.Context(local_rank)
        # every rank pins a host buffer for its whole result (16.4 GB): with many ranks on one box
        # keep the sum within the host's free memory (all ranks then use the same, smaller, number
        # of pairs for this leg; stated in the JSON line)
        n_e2e = n
        try:
            avail = next(int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable"))
            n_e2e = max(64, min(n, int(0.55 * avail / world) // (nx * ny * esz)))
        except Exception:
            pass
        if world > 1:
            tn = torch.tensor([n_e2e], device=dev, dtype=torch.int64)
            dist.all_reduce(tn, op=dist.ReduceOp.MIN)
            n_e2e = int(tn.item())
        n_full, n = n, n_e2e  # the e2e leg's batch
        src_full, smap_full = src, smap
        src = np.ascontiguousarray(src[:n])
        smap = None if smap is None else np.ascontiguousarray(smap[:n])
        cells_e2e = n * nx * ny
        out_h = torch.empty((n, ny, nx), dtype=tdt, pin_memory=True)  # (no pageable staging copy)
        out_np = out_h.numpy()
        lib, C = host_ctx.lib, __import__("ctypes")
        dt = vhp.F32 if args.store == "f32" else vhp.F64
        probe = sorted({0, n // 3, n // 2, n - 1})  # pairs checked against the device result

        def e2e_step():
            st = lib.vhp_visibility_batch(host_ctx.h, maps.ctypes.data, nmaps, nx, ny,
                                          src.ctypes.data, None if smap is None else smap.ctypes.data,
                                          n, dt, out_np.ctypes.data)
            assert st == 0, host_ctx.lib.vhp_last_error(host_ctx.h)

        def e2e_run(mode):
            host_ctx.set_result_transport(mode)
            e2e_step()  # warm-up (allocations, page mapping, host threads)
            for p in probe:
                out_np[p].fill(np.nan)  # the timed calls must rewrite them
            barrier()
            k = max(1, min(args.steps, 3))
            t0 = time.perf_counter()
            for _ in range(k):
                e2e_step()
            torch.cuda.synchronize()
            t = (time.perf_counter() - t0) / k
            if world > 1:
                tt = torch.tensor([t], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t = float(tt.item())
            for p in probe:
                assert np.array_equal(out_np[p], out_t[p].cpu().numpy()), f"e2e result differs (pair {p})"
            d2h, res, packed = host_ctx.last_transport()
            assert res == int(n) * nx * ny * esz
            return t, k, d2h, packed

        t_e2e, k_e2e, d2h_b, packed = e2e_run(1)   # the default (automatic) transport
        t_plain, _, d2h_plain, _ = e2e_run(0)      # plain copies, for comparison
        # the same call into an ordinary (pageable) caller buffer: the literal units are staged
        # through pinned memory and scattered by the host threads (bounded to 1024 pairs: the
        # buffer is touched for the first time inside the warm-up call)
        n_pg = min(n, 1024)
        out_pg = np.empty((n_pg, ny, nx), dtype=np.float32 if args.store == "f32" else np.float64)
        src_pg = np.ascontiguousarray(src[:n_pg])
        smap_pg = None if smap is None else np.ascontiguousarray(smap[:n_pg])

        def pg_step():
            st = lib.vhp_visibility_batch(host_ctx.h, maps.ctypes.data, nmaps, nx, ny, src_pg.ctypes.data,
                                          None if smap_pg is None else smap_pg.ctypes.data, n_pg, dt,
                                          out_pg.ctypes.data)
            assert st == 0, host_ctx.lib.vhp_last_error(host_ctx.h)
        host_ctx.set_result_transport(1)
        pg_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            pg_step()
        t_pg = (time.perf_counter() - t0) / 2
        if world > 1:
            tt = torch.tensor([t_pg], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_pg = float(tt.item())
        assert np.array_equal(out_pg[n_pg // 2], out_t[n_pg // 2].cpu().numpy())
        pageable = {"value": n_pg * nx * ny * world / t_pg / 1e9, "unit": "Gcells/s", "pairs_per_gpu": int(n_pg),
                    "ms_per_step": t_pg * 1e3, "transport": ["plain", "packed (staged literal stream)", "packed (direct)"][host_ctx.last_transport()[2]]}
        del out_pg
        e2e = {"value": cells_e2e * world / t_e2e / 1e9, "unit": "Gcells/s",
               "pairs_per_gpu": int(n),
               "h2d_bytes_per_step": int(maps.nbytes + src.nbytes + (0 if smap is None else smap.nbytes)),
               "d2h_bytes_per_step": int(d2h_b),
               "result_bytes_per_step": int(n) * nx * ny * esz,
               "ms_per_step": t_e2e * 1e3, "steps": k_e2e,
               "transport": ("packed%s: the device classifies 128-byte units of the results as uniform / "
                             "literal, %s; %s host threads write the uniform units; the host buffer is "
                             "bit-identical to the plain copy"
                             % (" (direct)" if packed == 2 else "",
                                "stores the literal units straight into the pinned host buffer" if packed == 2
                                else "the literal units are copied as one stream",
                                os.environ.get("VHP_HOST_THREADS", str(min(32, os.cpu_count() or 1)))))
                            if packed else "plain",
               "plain_transport": {"value": cells_e2e * world / t_plain / 1e9, "ms_per_step": t_plain * 1e3,
                                   "d2h_bytes_per_step": int(d2h_plain)},
               "pageable_buffer": pageable,
               "api": "vhp_visibility_batch (host buffers; pinned output; H2D + kernel + D2H (+ host expansion) "
                      "inside the timed region; %d result pairs compared with the device-resident run)" % len(probe)}
        # ---- the same fields as a packed handle (vhp_visibility_batch_packed): the lossless packed form
        # stays in pinned memory owned by the handle, pairs are expanded on demand
        ph = C.c_void_p()

        def packed_step():
            st = lib.vhp_visibility_batch_packed(host_ctx.h, maps.ctypes.data, nmaps, nx, ny, src.ctypes.data,
                                                 None if smap is None else smap.ctypes.data, n, dt, C.byref(ph))
            assert st == 0, host_ctx.lib.vhp_last_error(host_ctx.h)
        packed_step()  # (allocates the handle's pinned memory; later calls reuse it)
        barrier()
        kp = max(1, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(kp):
            packed_step()
        t_ph = (time.perf_counter() - t0) / kp
        if world > 1:
            tt = torch.tensor([t_ph], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_ph = float(tt.item())
        one = np.empty((ny, nx), dtype=out_np.dtype)
        t_x = 0.0
        for p_ in probe:  # lazy expansion of single pairs: the bytes of the device-resident run
            tx0 = time.perf_counter()
            st = lib.vhp_packed_expand(ph, int(p_), 1, one.ctypes.data, 1)
            t_x += time.perf_counter() - tx0
            assert st == 0 and np.array_equal(one, out_t[p_].cpu().numpy()), f"packed handle differs (pair {p_})"
        e2e["packed_handle"] = {"value": cells_e2e * world / t_ph / 1e9, "unit": "Gcells/s", "ms_per_step": t_ph * 1e3,
                                "steps": kp, "h2d_bytes_per_step": e2e["h2d_bytes_per_step"],
                                "d2h_bytes_per_step": int(lib.vhp_packed_bytes(ph)),
                                "result_bytes_per_step": int(n) * nx * ny * esz,
                                "expand_one_pair_ms": t_x / len(probe) * 1e3,
                                "api": "vhp_visibility_batch_packed (host buffers; H2D, sweeps, packing and the D2H of "
                                       "the packed stream into the handle's pinned memory inside the timed region; "
                                       "nothing is expanded in the call) + vhp_packed_expand of the probe pairs "
                                       "afterwards, bit-identical to the device-resident fields"}
        lib.vhp_packed_destroy(ph)
        # ---- the same call with the thresholded, bit-packed result (vhp_visibility_batch_bin)
        # (checked against the fp64 fields of the probe pairs: an fp32 value can sit on the other side
        # of the threshold)
        probe_src = torch.from_numpy(np.ascontiguousarray(src[probe])).to(dev)
        probe_map = None if smap is None else torch.from_numpy(np.ascontiguousarray(smap[probe])).to(dev)
        probe64 = torch.empty((len(probe), ny, nx), dtype=torch.float64, device=dev)
        with torch.cuda.stream(stream):
            ctx.visibility_batch_dev(occ_t, probe_src, probe64, probe_map)
        stream.synchronize()
        probe64 = {p_: probe64[k].cpu().numpy() for k, p_ in enumerate(probe)}
        wpr = (nx + 31) // 32
        bits_h = torch.empty((n, ny, wpr), dtype=torch.int32, pin_memory=True)
        bits_np = bits_h.numpy().view(np.uint32)
        thr_bin = 0.5

        def bin_step():
            st = lib.vhp_visibility_batch_bin(host_ctx.h, maps.ctypes.data, nmaps, nx, ny, src.ctypes.data,
                                              None if smap is None else smap.ctypes.data, n, thr_bin,
                                              bits_np.ctypes.data)
            assert st == 0, host_ctx.lib.vhp_last_error(host_ctx.h)
        bin_step()
        for p_ in probe:
            bits_np[p_].fill(0xA5A5A5A5)
        barrier()
        kb = max(1, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(kb):
            bin_step()
        torch.cuda.synchronize()
        t_bin = (time.perf_counter() - t0) / kb
        if world > 1:
            tt = torch.tensor([t_bin], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_bin = float(tt.item())
        for p_ in probe:
            assert np.array_equal(vhp.unpack_bits(bits_np[p_], nx), probe64[p_] >= thr_bin), f"binary e2e result differs (pair {p_})"
        e2e["binary"] = {"value": cells_e2e * world / t_bin / 1e9, "unit": "Gcells/s", "ms_per_step": t_bin * 1e3,
                         "steps": kb, "threshold": thr_bin,
                         "h2d_bytes_per_step": e2e["h2d_bytes_per_step"],
                         "d2h_bytes_per_step": int(n) * ny * wpr * 4,
                         "api": "vhp_visibility_batch_bin (host buffers, pinned output): H2D, sweeps that compare in fp64 "
                                "and write bits themselves (the field is never stored), D2H of 1 bit per cell, all inside "
                                "the timed region; bit-exact against the fp64 field compared with >= threshold "
                                "(tests/test_gpu_sweep.py)"}
        del bits_h
        # ---- ... and as row runs (vhp_visibility_batch_runs): transition columns per row
        rc_h = torch.empty((n, ny), dtype=torch.int16, pin_memory=True)
        pp_h = torch.empty(n + 1, dtype=torch.int64, pin_memory=True)
        cap = 16 * n * ny
        tr_h = torch.empty(cap, dtype=torch.int16, pin_memory=True)
        rc_np, pp_np, tr_np = rc_h.numpy().view(np.uint16), pp_h.numpy().view(np.uint64), tr_h.numpy().view(np.uint16)
        used = C.c_int64(0)

        def runs_step():
            st = lib.vhp_visibility_batch_runs(host_ctx.h, maps.ctypes.data, nmaps, nx, ny, src.ctypes.data,
                                               None if smap is None else smap.ctypes.data, n, thr_bin,
                                               rc_np.ctypes.data, pp_np.ctypes.data, tr_np.ctypes.data, cap,
                                               C.byref(used))
            assert st == 0, host_ctx.lib.vhp_last_error(host_ctx.h)
        runs_step()
        rc_np.fill(0)
        barrier()
        t0 = time.perf_counter()
        for _ in range(kb):
            runs_step()
        torch.cuda.synchronize()
        t_runs = (time.perf_counter() - t0) / kb
        if world > 1:
            tt = torch.tensor([t_runs], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_runs = float(tt.item())
        for p_ in probe:  # rebuild the probe pairs' bit maps from their runs
            lo, hi = int(pp_np[p_]), int(pp_np[p_ + 1])
            got = vhp.runs_to_bits(rc_np[p_:p_ + 1], np.array([0, hi - lo], np.uint64), tr_np[lo:hi], nx)[0]
            assert np.array_equal(vhp.unpack_bits(got, nx), probe64[p_] >= thr_bin), f"row runs differ (pair {p_})"
        d2h_runs, _, _ = host_ctx.last_transport()
        e2e["runs"] = {"value": cells_e2e * world / t_runs / 1e9, "unit": "Gcells/s", "ms_per_step": t_runs * 1e3,
                       "steps": kb, "threshold": thr_bin, "h2d_bytes_per_step": e2e["h2d_bytes_per_step"],
                       "d2h_bytes_per_step": int(d2h_runs), "transition_columns": int(pp_np[n]),
                       "api": "vhp_visibility_batch_runs (host buffers, pinned outputs): H2D, sweeps that write bits "
                              "themselves, run encoding on the device (transition columns per row), D2H, all inside the "
                              "timed region; bit-exact against the fp64 field compared with >= threshold "
                              "(tests/test_gpu_sweep.py)"}
        del rc_h, pp_h, tr_h
        n, src, smap = n_full, src_full, smap_full

    # ---- the same grid and batch size with obstacles (kernel-only, rank-local): how the
    # headline kernel does once the sweep is more than a fill -- reported beside the headline
    penumbra = None
    if args.workload == "c2" and not args.no_penumbra and not args.pairs:
        penumbra = {}
        for wl in ("c2s", "c2d", "c4"):
            m2, s2, sm2, d2 = workload(wl, rank, world)
            n2, (ny2, nx2) = len(s2), m2.shape[1:]
            o2 = torch.empty((n2, ny2, nx2), dtype=tdt, device=dev)
            occ2, src2 = torch.from_numpy(m2).to(dev), torch.from_numpy(s2).to(dev)
            smap2 = None if sm2 is None else torch.from_numpy(sm2).to(dev)
            with torch.cuda.stream(stream):
                ctx.prepare_maps_dev(occ2)
            ms = _timed_dev(stream, lambda: ctx.visibility_batch_dev(occ2, src2, o2, smap2), 10)
            byts = n2 * nx2 * ny2 * esz + m2.shape[0] * nx2 * ny2
            penumbra[wl] = {"workload": d2, "ms_per_step": ms, "value": n2 * nx2 * ny2 / ms / 1e6,
                            "unit": "Gcells/s", "achieved_gbs": byts / ms / 1e6,
                            "frac_of_hbm_peak": byts / ms / 1e6 / measured_peak()[0], "steps": 10}
            if wl == "c2s" and e2e is not None and tuple(o2.shape) == tuple(out_np.shape):
                # the same host-buffer call on the obstacle workload (automatic transport)
                def c2s_step():
                    st = lib.vhp_visibility_batch(host_ctx.h, m2.ctypes.data, m2.shape[0], nx2, ny2,
                                                  s2.ctypes.data, None, n2, dt, out_np.ctypes.data)
                    assert st == 0, host_ctx.lib.vhp_last_error(host_ctx.h)
                host_ctx.set_result_transport(1)
                c2s_step()
                for p in probe:
                    out_np[p].fill(np.nan)
                t0 = time.perf_counter()
                for _ in range(2):
                    c2s_step()
                t2 = (time.perf_counter() - t0) / 2
                for p in probe:
                    assert np.array_equal(out_np[p], o2[p].cpu().numpy()), f"c2s e2e result differs (pair {p})"
                d2h2, res2, packed2 = host_ctx.last_transport()
                penumbra[wl]["e2e"] = {"value": n2 * nx2 * ny2 / t2 / 1e9, "unit": "Gcells/s",
                                       "ms_per_step": t2 * 1e3, "d2h_bytes_per_step": int(d2h2),
                                       "result_bytes_per_step": int(res2),
                                       "transport": ["plain", "packed", "packed (direct)"][packed2], "steps": 2}
            del o2
            # the same batch as thresholded bits (the sweep writes 1 bit per cell, nothing else)
            ob = torch.empty((n2, ny2, (nx2 + 31) // 32), dtype=torch.int32, device=dev)
            msb = _timed_dev(stream, lambda: ctx.visibility_batch_bin_dev(occ2, src2, 0.5, ob, smap2), 5)
            penumbra[wl]["bits_store"] = {"ms_per_step": msb, "value": n2 * nx2 * ny2 / msb / 1e6, "unit": "Gcells/s",
                                          "threshold": 0.5}
            del ob
            if wl in ("c2s", "c2d") and args.store == "f32":  # the same batch stored as fp64 (north_star's fp64 mode)
                o3 = torch.empty((n2, ny2, nx2), dtype=torch.float64, device=dev)
                ms3 = _timed_dev(stream, lambda: ctx.visibility_batch_dev(occ2, src2, o3, smap2), 5)
                b3 = n2 * nx2 * ny2 * 8 + m2.shape[0] * nx2 * ny2
                penumbra[wl]["f64_store"] = {"ms_per_step": ms3, "value": n2 * nx2 * ny2 / ms3 / 1e6, "unit": "Gcells/s",
                                             "achieved_gbs": b3 / ms3 / 1e6,
                                             "frac_of_hbm_peak": b3 / ms3 / 1e6 / measured_peak()[0]}
                del o3
            del occ2, src2
    f64_store = None
    if args.workload == "c2" and args.store == "f32" and not args.no_penumbra and not args.pairs:
        with torch.cuda.stream(stream):
            ctx.prepare_maps_dev(occ_t)
        o3 = torch.empty((n, ny, nx), dtype=torch.float64, device=dev)
        ms3 = _timed_dev(stream, lambda: ctx.visibility_batch_dev(occ_t, src_t, o3, smap_t), 10)
        b3 = n * nx * ny * 8 + nmaps * nx * ny
        f64_store = {"workload": "the headline batch stored as fp64 (bit-identical to the reference's Field<double>)",
                     "ms_per_step": ms3, "value": cells / ms3 / 1e6, "unit": "Gcells/s",
                     "roofline": {"bound": "hbm", "achieved": b3 / ms3 / 1e6, "peak": measured_peak()[0], "unit": "GB/s",
                                  "frac": b3 / ms3 / 1e6 / measured_peak()[0], "algorithmic_bytes_per_launch": b3}}
        del o3
        ob = torch.empty((n, ny, (nx + 31) // 32), dtype=torch.int32, device=dev)
        msb = _timed_dev(stream, lambda: ctx.visibility_batch_bin_dev(occ_t, src_t, 0.5, ob, smap_t), 10)
        f64_store["bits_store"] = {"workload": "the headline batch as thresholded bits (vhp_visibility_batch_bin_dev: "
                                               "the sweep compares in fp64 and writes 1 bit per cell)",
                                   "ms_per_step": msb, "value": cells / msb / 1e6, "unit": "Gcells/s", "threshold": 0.5}
        del ob
    if e2e is not None:
        host_ctx.close()
        del out_h

    # ---- BASELINE configs[4]: one dense 8192 x 8192 map, the planner over all ranks (strip
    # partition, NCCL inside the library); not part of `value`
    giant = None
    if args.workload == "c2" and not args.no_giant and not args.pairs:
        giant = giant_leg(vhp, local_rank, rank, world, dist if world > 1 else None)

    # ---- single-GPU latency / comparison legs of the other BASELINE configs (rank 0, N = 1)
    c1 = c3 = raycast = None
    if args.workload == "c2" and world == 1 and not args.pairs and not args.no_legs:
        c1 = c1_leg(vhp, ctx, stream, dev, local_rank, not args.no_cpu)
        c3 = c3_leg(vhp, local_rank, not args.no_cpu)
        raycast = raycast_leg(vhp, ctx, stream, dev, not args.no_cpu)

    planner = None
    if not args.no_planner:
        planner = planner_leg(vhp, local_rank, rank, world, dist if world > 1 else None, dev,
                              not args.no_cpu and world == 1)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    alg_bytes = n * nx * ny * esz + nmaps * nx * ny  # stores + each map read once
    kern_ms = statistics.mean(step_ms)
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu_traffic(args.workload, n) if args.store == "f32" else None,  # the captures are of the fp32 kernel
                "kernel": "sweep_tile_kernel", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "traffic_source": "profiles/k1_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum per pair; "
                                  "null unless that capture was taken from the kernel sources benchmarked here, hash %s)"
                                  % kernel_source_hash(),
                "note": "per-launch time = CUDA events around one step on the launch stream "
                        "(one sweep kernel per step; the maps' bit planes are packed before the timed region); the peak is the "
                        "driver's STREAM-copy figure, a write-only stream can exceed it (torch fill_ of the "
                        "same buffer: 7.5 TB/s on this pool)"}
    cpu = None
    if not args.no_cpu and world == 1:
        cpu = cpu_baseline(maps, src, nx, ny)
    line = {"metric": METRIC, "value": value, "unit": "Gcells/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.workload, desc, nx, ny, n, args.store, world), "rank0_numa_node": numa_node,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches), "planner": planner, "penumbra": penumbra, "f64_store": f64_store,
            "giant": giant, "c1": c1, "c3": c3, "raycast": raycast}
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
