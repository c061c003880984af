"""Midgame search throughput (othello_search) on one GPU, with a one-core CPU figure for the same positions.

    python tools/bench_search.py [--empties 44,34,24] [--depths 2,4,6,8] [--count 20000] [--cpu 50] [--seed 4]

Positions with exactly E empty squares come from seeded random playouts on the GPU (ops.playout): the first position
of each game that has E empties, in game order, so the sample is fixed by the seed and two builds search the same set.
Per (table, E, depth): one JSON line with the positions, kernel time (CUDA events around ops.search, after one warm-up
call of the same shape), positions/s, nodes/s, mean and max nodes per position, and the host build of
csrc/midgame.cuh (tests/search_host.cpp, compiled into a temporary directory) on the first --cpu positions on one
core, whose results must equal the kernel's bit for bit.  Two tables: default_value() and a learnt-looking integer
table.  GPU name, power limit and SM clocks are read with nvidia-smi (queries only) in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from subproc_b200 import ops  # noqa: E402
from bench_solve import gpu_info, positions  # noqa: E402

# default_value() (parameter_progress_position_moves_learn.py:30-36) and a table shaped like a learnt one: corners and
# mobility high, X- and C-squares negative, intercepts non-zero
TABLES = {
    "default": [[100, 99, -1, -1, -1, -1, 3, 8, 20, 0], [75, 99, 2, -5, 7, 6, 4, 5, 5, 0],
                [25, 99, 2, -5, -7, -6, 4, 5, 5, 0], [1, 100, 50, 30, 30, 30, 30, 30, 30, 0]],
    "learnt": [[12, 61, -38, -17, 9, 4, -2, 3, 1, -6], [15, 57, -29, -12, 6, 3, -1, 2, 2, -4],
               [11, 48, -18, -8, 5, 4, 1, 3, 2, 3], [4, 39, -6, -3, 4, 5, 3, 4, 3, 9]],
}


def host_searcher():
    out = os.path.join(tempfile.mkdtemp(prefix="bench_search_"), "search_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++",
                           os.path.join(ROOT, "tests", "search_host.cpp"), "-o", out])
    return ctypes.CDLL(out)


def host_search(L, b, w, t, weights, depth):
    n = b.size
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    b, w, t = np.ascontiguousarray(b), np.ascontiguousarray(w), np.ascontiguousarray(t)
    v, m, nodes = np.zeros(n, np.float32), np.zeros(n, np.uint8), np.zeros(n, np.uint64)
    t0 = time.perf_counter()
    L.mg_search(p(b), p(w), p(t), p(weights), ctypes.c_int(depth), p(v), p(m), p(nodes), ctypes.c_long(n))
    return time.perf_counter() - t0, v, m, nodes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--empties", default="44,34,24")
    ap.add_argument("--depths", default="2,4,6,8")
    ap.add_argument("--count", type=int, default=20000, help="positions searched per (E, depth)")
    ap.add_argument("--cpu", type=int, default=50, help="positions of those the host build searches on one core")
    ap.add_argument("--seed", type=int, default=4)
    ap.add_argument("--games", type=int, default=1 << 15)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_search needs a CUDA device"
    dev = torch.device("cuda:0")
    info = gpu_info()
    L = host_searcher()
    for name, rows in TABLES.items():
        wh = np.ascontiguousarray(np.asarray(rows, np.float32))
        wd = torch.from_numpy(wh).to(dev)
        for e in [int(x) for x in args.empties.split(",")]:
            b, w, t = positions(e, args.games, args.seed + e, dev)
            n = min(args.count, b.size)
            b, w, t = b[:n], w[:n], t[:n]
            db, dw, dt = ops.bits_tensor(b, dev), ops.bits_tensor(w, dev), torch.from_numpy(t).to(dev)
            for depth in [int(x) for x in args.depths.split(",")]:
                ops.search(db, dw, wd, depth, turn=dt, nodes=True)             # warm-up: module load, first launch
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                v, m, nodes = ops.search(db, dw, wd, depth, turn=dt, nodes=True)
                e1.record()
                e1.synchronize()
                sec = e0.elapsed_time(e1) * 1e-3
                nodes = nodes.cpu().numpy()
                k = min(args.cpu, n)
                cpu_sec, hv, hm, hn = host_search(L, b[:k], w[:k], t[:k], wh, depth)
                assert np.array_equal(hv.view(np.uint32), v.cpu().numpy()[:k].view(np.uint32))
                assert np.array_equal(hm, m.cpu().numpy()[:k]) and np.array_equal(hn.astype(np.int64), nodes[:k])
                print(json.dumps({
                    "table": name, "empties": e, "depth": depth, "positions": int(n), "kernel_s": round(sec, 4),
                    "positions_per_s": n / sec, "nodes_per_s": float(nodes.sum()) / sec,
                    "nodes_mean": float(nodes.mean()), "nodes_max": int(nodes.max()),
                    "cpu_positions": int(k), "cpu_s": round(cpu_sec, 3), "cpu_positions_per_s": k / cpu_sec,
                    "cpu_nodes_per_s": float(hn.sum()) / cpu_sec, "cpu_cores_used": 1, "cpu_cores": os.cpu_count(),
                    "gpu": info, "seed": args.seed + e}), flush=True)


if __name__ == "__main__":
    main()
