"""The strip-partitioned planner across GPUs: one rank per GPU, halo rows by ncclSend / ncclRecv and
the arg-min key by ncclAllGather inside the library (csrc/giant.cu).  Runs tools/giant_multi_gpu.py
under torch.distributed.run on 2 GPUs (and on every GPU of the box): every rank compares its rows of
the fields, the light sources and the path with the single-GPU planner, bit for bit.  Skipped on a
box with one GPU (the single-process strips of tests/test_gpu_giant.py still run there)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    import torch
    return torch.cuda.device_count()


def _run(nproc, size, queries, spr=1, port=29541, p2p=True, map_kind="random"):
    env = dict(os.environ)
    env["VHP_GIANT_P2P"] = "1" if p2p else "0"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tools", "giant_multi_gpu.py"), "--size", str(size), "--queries", str(queries),
           "--spr", str(spr), "--max-iter", "40", "--map", map_kind]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def test_two_ranks_equal_single_gpu():
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    # strip boundaries tile by tile through peer memory (NVLink stores inside the sweep kernels)
    r = _run(2, 1536, 3)
    assert r["all_ranks_equal"] and all(q["equal_single_gpu"] for q in r["queries"])
    assert all(q["peer_handover"] == 1 for q in r["queries"])
    # ... and as finished rows by ncclSend / ncclRecv
    r = _run(2, 1536, 3, port=29544, p2p=False)
    assert r["all_ranks_equal"] and all(q["equal_single_gpu"] for q in r["queries"])
    assert all(q["peer_handover"] == 0 and q["halo_bytes_sent"] > 0 for q in r["queries"] if q["iterations"] > 0)
    r = _run(2, 1024, 2, spr=3, port=29542)   # remote and local strip boundaries mixed (NCCL hand-over)
    assert r["all_ranks_equal"]


def test_two_ranks_ties_across_the_rank_boundary():
    """A map mirrored about both axes, the middle row rank 0's last: cells mirrored about the start's row tie on
    h and lie on different ranks, so the all-gathered minimum has to keep the first pushed (peer memory and NCCL)"""
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    for port, p2p in ((29546, True), (29547, False)):
        r = _run(2, 1024, 4, port=port, p2p=p2p, map_kind="mirrored")
        assert r["n"] == 1025 and r["all_ranks_equal"] and all(q["equal_single_gpu"] for q in r["queries"])


def test_all_gpus_equal_single_gpu():
    n = _gpus()
    if n < 4:
        pytest.skip("needs >= 4 GPUs")
    r = _run(n, 4096, 2, port=29543)
    assert r["all_ranks_equal"] and all(q["equal_single_gpu"] for q in r["queries"])
    r = _run(n, 4096, 2, port=29545, p2p=False)
    assert r["all_ranks_equal"] and all(q["equal_single_gpu"] for q in r["queries"])


def test_sharded_batch_equals_single_gpu():
    """SURVEY 4 item iv on hardware: a (map, source) batch and a planner batch cut over the GPUs of the
    box (sharding.py, no data-path collective) give, item for item, the bytes one GPU computes for the
    whole batch (fp64 fields, thresholded bits, planner outputs; tools/sharded_batch_gpu.py)."""
    n = _gpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29551", os.path.join(ROOT, "tools", "sharded_batch_gpu.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    r = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert r["world"] == n and r["sweeps_equal"] and r["planner_equal"], r
