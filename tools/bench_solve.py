"""Exact endgame solver throughput (othello_solve) on one GPU, with a one-core CPU figure for the same positions.

    python tools/bench_solve.py [--empties 12,16,20] [--count 12:20000,16:256,20:1] [--cpu 12:200,16:8,20:1] [--seed 4]

Positions with exactly E empty squares come from seeded random playouts on the GPU (ops.playout): the first position
of each game that has E empties, in game order, so the sample is fixed by the seed and two builds solve the same set.
Per E: one JSON line with the positions, kernel time (CUDA events around ops.solve, after one warm-up call), positions/s,
nodes/s, mean and max nodes per position, and the host build of csrc/endgame.cuh (tests/solve_host.cpp, compiled by
tests/host_build.py) on the first --cpu positions on one core.  A call at E empties lasts as long as its slowest
position (one lane solves one position), so the counts shrink with E.  GPU name, power limit and SM clocks are read
with nvidia-smi (queries only) in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from subproc_b200 import ops  # noqa: E402
import host_build  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"name": torch.cuda.get_device_name(0)}


def popcount(x):
    x = x - ((x >> np.uint64(1)) & np.uint64(0x5555555555555555))
    x = (x & np.uint64(0x3333333333333333)) + ((x >> np.uint64(2)) & np.uint64(0x3333333333333333))
    x = (x + (x >> np.uint64(4))) & np.uint64(0x0F0F0F0F0F0F0F0F)
    return ((x * np.uint64(0x0101010101010101)) >> np.uint64(56)).astype(np.int64)


def positions(empties, n_games, seed, dev):
    """black, white, turn (numpy) of the first position with `empties` empties in each seeded random playout"""
    po = ops.playout(n_games, seed=seed, device=dev)
    occ = (po.black | po.white).cpu().numpy().view(np.uint64)                       # [t_max+1][n]
    cnt = popcount(occ)
    nplies = po.nplies.cpu().numpy()
    valid = np.arange(occ.shape[0])[:, None] <= nplies[None, :]
    hit = (64 - cnt == empties) & valid
    games = np.nonzero(hit.any(0))[0]
    t = hit[:, games].argmax(0)
    b = ops.bits_numpy(po.black)[t, games]
    w = ops.bits_numpy(po.white)[t, games]
    turn = np.where(t % 2 == 0, ops.BLACK, ops.WHITE).astype(np.uint8)
    return b, w, turn


def host_solve(L, b, w, t):
    n = b.size
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    b, w, t = np.ascontiguousarray(b), np.ascontiguousarray(w), np.ascontiguousarray(t)
    v, m, nodes = np.zeros(n, np.int32), np.zeros(n, np.uint8), np.zeros(n, np.uint64)
    t0 = time.perf_counter()
    L.eg_solve(p(b), p(w), p(t), p(v), p(m), p(nodes), ctypes.c_long(n))
    return time.perf_counter() - t0, v, m, nodes


def per_e(arg, default):
    d = dict(default)
    for kv in filter(None, arg.split(",")):
        k, v = kv.split(":")
        d[int(k)] = int(v)
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--empties", default="12,16,20")
    ap.add_argument("--count", default="", help="E:n,... positions solved per E")
    ap.add_argument("--cpu", default="", help="E:n,... positions of those the host build solves on one core")
    ap.add_argument("--seed", type=int, default=4)
    ap.add_argument("--games", type=int, default=1 << 15)
    args = ap.parse_args()
    count = per_e(args.count, {12: 20000, 16: 256, 20: 1})
    ncpu = per_e(args.cpu, {12: 200, 16: 8, 20: 1})
    assert torch.cuda.is_available(), "bench_solve needs a CUDA device"
    dev = torch.device("cuda:0")
    info = gpu_info()
    L = host_build.load("solve_host.cpp")
    warm = True
    for e in [int(x) for x in args.empties.split(",")]:
        b, w, t = positions(e, args.games, args.seed + e, dev)
        n = min(count.get(e, 100), b.size)
        b, w, t = b[:n], w[:n], t[:n]
        db, dw, dt = ops.bits_tensor(b, dev), ops.bits_tensor(w, dev), torch.from_numpy(t).to(dev)
        if warm:                                                   # module load, first launch
            ops.solve(db[:256], dw[:256], dt[:256], nodes=True)
            torch.cuda.synchronize()
            warm = False
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        v, m, nodes = ops.solve(db, dw, dt, nodes=True)
        e1.record()
        e1.synchronize()
        sec = e0.elapsed_time(e1) * 1e-3
        nodes = nodes.cpu().numpy()
        k = min(ncpu.get(e, 1), n)
        cpu_sec, hv, hm, hn = host_solve(L, b[:k], w[:k], t[:k])
        assert np.array_equal(hv, v.cpu().numpy()[:k]) and np.array_equal(hm, m.cpu().numpy()[:k])
        assert np.array_equal(hn.astype(np.int64), nodes[:k])
        print(json.dumps({
            "empties": e, "positions": int(n), "kernel_s": round(sec, 4), "positions_per_s": n / sec,
            "nodes_per_s": float(nodes.sum()) / sec, "nodes_mean": float(nodes.mean()), "nodes_max": int(nodes.max()),
            "cpu_positions": int(k), "cpu_s": round(cpu_sec, 3), "cpu_positions_per_s": k / cpu_sec,
            "cpu_nodes_per_s": float(hn.sum()) / cpu_sec, "cpu_cores_used": 1, "cpu_cores": os.cpu_count(),
            "gpu": info, "seed": args.seed + e}), flush=True)


if __name__ == "__main__":
    main()
