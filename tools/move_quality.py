"""How good a table's moves are, without playing a match: the disc loss of an engine's move against perfect play.

    python tools/move_quality.py [--empties 14,18,20] [--count 14:4096,18:512,20:128] [--depths 1,2,4,6] [--seed 12]

Positions with exactly E empty squares come from seeded greedy self-play on default_value() with 10 random plies (the
first position of each game that has E empties, in game order); only positions where the mover has at least two
legal moves are kept, so every engine has a choice.  ops.solve_moves scores every move of every position exactly.
For each table (default_value() and the learnt-looking table of tools/bench_search.py) and each engine (the move
ops.search returns at depth 1 = greedy, 2, 4, 6 on that table), and for a uniformly random legal move as a baseline:
one JSON line per (table, engine, E) with the mean disc loss of the engine's move against the best move (the best
move's value minus the played move's, from the mover's side, empties not given to the winner) and the share of
positions where the engine's move is a perfect one (loss 0).  GPU name, power limit and SM clocks are read with
nvidia-smi (queries only) in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from subproc_b200 import ops  # noqa: E402
from bench_solve import gpu_info, per_e, popcount  # noqa: E402
from bench_search import TABLES  # noqa: E402


def greedy_positions(empties, n_games, seed, weights, dev):
    """black, white, turn (device) of the first position with `empties` empties in each seeded greedy game"""
    po = ops.playout(n_games, seed=seed, device=dev, policy=ops.POLICY_GREEDY, random_plies=10, weights=weights)
    occ = (po.black | po.white).cpu().numpy().view(np.uint64)
    valid = np.arange(occ.shape[0])[:, None] <= po.nplies.cpu().numpy()[None, :]
    hit = (64 - popcount(occ) == empties) & valid
    games = np.nonzero(hit.any(0))[0]
    t = hit[:, games].argmax(0)
    b, w = ops.bits_numpy(po.black)[t, games], ops.bits_numpy(po.white)[t, games]
    turn = np.where(t % 2 == 0, ops.BLACK, ops.WHITE).astype(np.uint8)
    return ops.bits_tensor(b, dev), ops.bits_tensor(w, dev), torch.from_numpy(turn).to(dev)


def line(table, engine, depth, e, loss, info, seed):
    return json.dumps({"table": table, "engine": engine, "depth": depth, "empties": e, "positions": int(loss.numel()),
                       "mean_disc_loss": float(loss.float().mean()), "perfect_share": float((loss == 0).float().mean()),
                       "gpu": info, "seed": seed})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--empties", default="14,18,20")
    ap.add_argument("--count", default="", help="E:n,... positions sampled per E (before keeping those with a choice)")
    ap.add_argument("--depths", default="1,2,4,6")
    ap.add_argument("--seed", type=int, default=12)
    ap.add_argument("--games", type=int, default=1 << 14)
    args = ap.parse_args()
    count = per_e(args.count, {14: 4096, 18: 512, 20: 128})
    assert torch.cuda.is_available(), "move_quality needs a CUDA device"
    dev = torch.device("cuda:0")
    info = gpu_info()
    tables = {name: torch.tensor(rows, dtype=torch.float32, device=dev) for name, rows in TABLES.items()}
    gen = torch.Generator(device=dev)
    for e in [int(x) for x in args.empties.split(",")]:
        b, w, t = greedy_positions(e, args.games, args.seed + e, tables["default"], dev)
        n = min(count.get(e, 128), b.numel())
        values, _ = ops.solve_moves(b[:n].contiguous(), w[:n].contiguous(), turn=t[:n].contiguous())
        legal = values[:, :64] != ops.SOLVE_REFUSED
        keep = legal.sum(dim=1) >= 2
        b, w, t, values, legal = (x[:n][keep].contiguous() for x in (b, w, t, values, legal))
        best = values[:, :64].masked_fill(~legal, -1000).max(dim=1).values
        rows = torch.arange(b.numel(), device=dev)
        gen.manual_seed(args.seed + e)
        pick = torch.rand(legal.shape, generator=gen, device=dev).masked_fill(~legal, -1.0).argmax(dim=1)
        print(line(None, "random", 0, e, best - values[rows, pick], info, args.seed + e), flush=True)
        for name, wt in tables.items():
            for depth in [int(x) for x in args.depths.split(",")]:
                _, move, _ = ops.search(b, w, wt, depth, turn=t)
                engine = "greedy" if depth == 1 else "search"
                print(line(name, engine, depth, e, best - values[rows, move.long()], info, args.seed + e), flush=True)


if __name__ == "__main__":
    main()
