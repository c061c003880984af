"""Move-value throughput (othello_search_moves, othello_solve_moves) on one GPU, against othello_search / othello_solve
on the same positions.

    python tools/bench_move_values.py [--empties 44,34,24] [--depths 2,4,6] [--count 20000]
                                      [--solve-empties 12,16,20] [--solve-count 12:20000,16:64,20:1] [--seed 4]

Positions with exactly E empty squares come from seeded random playouts on the GPU, as in tools/bench_search.py and
tools/bench_solve.py (the first position of each game that has E empties), so the sample is fixed by the seed.  One
JSON line per case: search cases per (table, E, depth) on the two tables of bench_search.py, solver cases per E.  Each
line has the positions, the move values computed (entries that are not NaN / REFUSED), the kernel time (CUDA events
around one call, after a warm-up call of the same shape), positions/s, move values/s and nodes/s, the same positions'
ops.search / ops.solve time (measured the same way) with the ratio, and whether every row's maximum and lowest arg-max
agreed with ops.search / ops.solve.  A call lasts as long as its slowest move (one lane per move), so the solver
counts shrink with E.  GPU name, power limit and SM clocks are read with nvidia-smi (queries only) in the same run.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from subproc_b200 import ops  # noqa: E402
from bench_solve import gpu_info, per_e, positions  # noqa: E402
from bench_search import TABLES  # noqa: E402


def timed(fn):
    """fn() once to warm up, then once between CUDA events: (seconds, result)"""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3, out


def row_max(values, has):
    """(max, lowest arg-max, row has a value) of [n][65] rows whose entries `has` are values"""
    low = torch.full_like(values, -float("inf") if values.is_floating_point() else -1000)
    v = torch.where(has, values, low)
    arg = torch.argmax(v, dim=1)                   # the first maximum: the lowest index reaching it
    return v.gather(1, arg[:, None])[:, 0], arg, has.any(dim=1)


def agree(values, has, value, move):
    best, arg, any_ = row_max(values, has)
    rooted = move != ops.NO_MOVE
    bits = (lambda x: x.view(torch.int32)) if values.is_floating_point() else (lambda x: x)
    same_value = bits(best[rooted]) == bits(value[rooted])
    return bool(torch.equal(any_, rooted) and same_value.all() and (arg[rooted].to(torch.uint8) == move[rooted]).all())


def report(line, n, sec, ref_sec, has, nodes, info, seed):
    k = int(has.sum())
    line.update({"positions": int(n), "move_values": k, "kernel_s": round(sec, 4), "positions_per_s": n / sec,
                 "move_values_per_s": k / sec, "nodes_per_s": float(nodes.sum()) / sec,
                 "nodes_per_move_mean": float(nodes.sum()) / max(k, 1), "nodes_per_move_max": int(nodes.max()),
                 "reference_s": round(ref_sec, 4), "time_over_reference": sec / ref_sec, "gpu": info, "seed": seed})
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--empties", default="44,34,24")
    ap.add_argument("--depths", default="2,4,6")
    ap.add_argument("--count", type=int, default=20000, help="positions per search case")
    ap.add_argument("--solve-empties", default="12,16,20")
    ap.add_argument("--solve-count", default="", help="E:n,... positions per solver case")
    ap.add_argument("--seed", type=int, default=4)
    ap.add_argument("--games", type=int, default=1 << 15)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_move_values needs a CUDA device"
    dev = torch.device("cuda:0")
    info = gpu_info()
    for name, rows in TABLES.items():
        wd = torch.tensor(rows, dtype=torch.float32, device=dev)
        for e in [int(x) for x in args.empties.split(",") if x]:
            b, w, t = positions(e, args.games, args.seed + e, dev)
            n = min(args.count, b.size)
            db, dw, dt = ops.bits_tensor(b[:n], dev), ops.bits_tensor(w[:n], dev), torch.from_numpy(t[:n]).to(dev)
            for depth in [int(x) for x in args.depths.split(",")]:
                sec, (values, nodes) = timed(lambda: ops.search_moves(db, dw, wd, depth, turn=dt, nodes=True))
                ref_sec, (value, move, _) = timed(lambda: ops.search(db, dw, wd, depth, turn=dt))
                has = ~torch.isnan(values)
                line = {"kind": "search", "table": name, "empties": e, "depth": depth,
                        "agrees_with_search": agree(values, has, value, move)}
                report(line, n, sec, ref_sec, has, nodes, info, args.seed + e)
    count = per_e(args.solve_count, {12: 20000, 16: 64, 20: 1})
    for e in [int(x) for x in args.solve_empties.split(",") if x]:
        b, w, t = positions(e, args.games, args.seed + e, dev)
        n = min(count.get(e, 100), b.size)
        db, dw, dt = ops.bits_tensor(b[:n], dev), ops.bits_tensor(w[:n], dev), torch.from_numpy(t[:n]).to(dev)
        sec, (values, nodes) = timed(lambda: ops.solve_moves(db, dw, turn=dt, nodes=True))
        ref_sec, (value, move, _) = timed(lambda: ops.solve(db, dw, dt))
        has = values != ops.SOLVE_REFUSED
        line = {"kind": "solve", "empties": e, "agrees_with_solve": agree(values, has, value, move)}
        report(line, n, sec, ref_sec, has, nodes, info, args.seed + e)


if __name__ == "__main__":
    main()
