"""Match a search engine against the greedy engine, or against a second table, from a sample of openings.

    python tools/match_search.py [--depths 2,4,6] [--openings 4096] [--table default] [--opponent greedy] [--seed 8]

Openings are a seeded sample of distinct positions after 8 random plies from the standard opening (the leaves of the
opening book).  Each opening is played twice with the colours swapped (game_runner.play_search_games, lock-step on the
GPU): ``--table`` searched to depth D against ``--opponent`` -- 'greedy' (the same table, depth 1) or the name of a
second table of tools/bench_search.py searched to the same depth.  Per depth: one JSON line with wins / draws / losses
of the searching side and its mean disc difference (own - opponent discs at the end, empties not counted), the GPU
name, power limit and clocks.  This measures whether deeper search, or a table, plays stronger.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from subproc_b200 import ops  # noqa: E402
from subproc_b200.game_runner import play_search_games  # noqa: E402
from bench_search import TABLES  # noqa: E402
from bench_solve import gpu_info, popcount  # noqa: E402

BOOK_PLIES = 8


def openings(n, seed, dev):
    """n distinct positions after BOOK_PLIES random plies (Black to move: no game passes that early), seeded"""
    po = ops.playout(4 * n, seed=seed, device=dev, t_max=BOOK_PLIES)
    b, w = ops.bits_numpy(po.black[BOOK_PLIES]), ops.bits_numpy(po.white[BOOK_PLIES])
    pairs = np.unique(np.stack([b, w], 1), axis=0)
    pick = np.random.RandomState(seed).choice(len(pairs), n, replace=False)
    return pairs[pick, 0].copy(), pairs[pick, 1].copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depths", default="2,4,6")
    ap.add_argument("--openings", type=int, default=4096)
    ap.add_argument("--table", default="default", choices=sorted(TABLES))
    ap.add_argument("--opponent", default="greedy", choices=["greedy"] + sorted(TABLES))
    ap.add_argument("--seed", type=int, default=8)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "match_search needs a CUDA device"
    dev = torch.device("cuda:0")
    info = gpu_info()
    b, w = openings(args.openings, args.seed, dev)
    n = b.size
    b0, w0 = ops.bits_tensor(b, dev), ops.bits_tensor(w, dev)
    ta = torch.tensor(TABLES[args.table], dtype=torch.float32, device=dev)
    tb = torch.tensor(TABLES[args.table if args.opponent == "greedy" else args.opponent], dtype=torch.float32, device=dev)
    for depth in [int(x) for x in args.depths.split(",")]:
        d_opp = 1 if args.opponent == "greedy" else depth
        t0 = time.perf_counter()
        first = play_search_games(n, ta, depth, tb, d_opp, dev, black0=b0, white0=w0, trajectory=False)   # searcher Black
        second = play_search_games(n, tb, d_opp, ta, depth, dev, black0=b0, white0=w0, trajectory=False)  # ... White
        diff = lambda po: popcount(ops.bits_numpy(po.final_black)) - popcount(ops.bits_numpy(po.final_white))
        d = np.concatenate([diff(first), -diff(second)])
        sec = time.perf_counter() - t0
        print(json.dumps({
            "table": args.table, "depth": depth, "opponent": args.opponent, "opponent_depth": d_opp,
            "openings": int(n), "games": int(d.size), "wins": int((d > 0).sum()), "draws": int((d == 0).sum()),
            "losses": int((d < 0).sum()), "mean_disc_diff": round(float(d.mean()), 3), "wall_s": round(sec, 2),
            "gpu": info, "seed": args.seed}), flush=True)


if __name__ == "__main__":
    main()
