"""Search self-play throughput (othello_playout with OTHELLO_POLICY_SEARCH) on one GPU.

    python tools/bench_search_playout.py [--depths 1,2,4,6] [--games N,...] [--lock-step N,...] [--seed 1]

Per depth, one JSON line:
  * self-play from the standard opening with random_plies = 8 on default_value(): games/s, plies/s and searched
    positions/s (plies at t >= 8 whose mover had at least 2 legal moves: every ply that went to the search).  Kernel
    time by CUDA events around ops.playout, after a warm-up call of the same shape.
  * nodes/s: the searched positions are read back from the trajectories and searched again with ops.search(nodes=True);
    node counts are a function of (position, depth, weights), so their sum is what the kernel visited.
  * the same kind of games without random plies, from 8-ply openings: the kernel against play_search_games (lock-step
    from the host, one search launch per colour and ply).  Both must produce identical games; both times are reported
    (host clock around work that ends in a device synchronise, after a small warm-up call of each).
  * depth 1 only: the same games with POLICY_GREEDY (the greedy kernel), which must be identical, and its time.
GPU name, power limit and SM clocks are read with nvidia-smi (queries only) in the same run.
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from subproc_b200 import ops, parameter  # noqa: E402
from subproc_b200.game_runner import play_search_games  # noqa: E402
from bench_solve import gpu_info  # noqa: E402

RANDOM_PLIES = 8
GAMES = {1: 1 << 20, 2: 1 << 17, 4: 1 << 15, 6: 1 << 13}          # each call well over 0.1 s
LOCK_STEP = {1: 4096, 2: 4096, 4: 2048, 6: 1024}


def events_time(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3, out


def wall_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def same_games(a, b):
    """identical nplies, final positions, recorded rows t <= nplies and moves t < nplies"""
    if not (torch.equal(a.nplies, b.nplies) and torch.equal(a.final_black, b.final_black)
            and torch.equal(a.final_white, b.final_white)):
        return False
    t = torch.arange(a.t_max + 1, device=a.nplies.device)[:, None]
    n = a.nplies.long()[None, :]
    rows, moves = t <= n, t[:-1] < n
    return (torch.equal(a.black[rows], b.black[rows]) and torch.equal(a.white[rows], b.white[rows])
            and torch.equal(a.move[moves], b.move[moves]))


def searched_positions(po, first):
    """(own, opp) of every ply t >= first that had at least 2 legal moves (Black moves at even t: a pass is a ply)"""
    owns, opps = [], []
    for t in range(first, int(po.nplies.max()) + 1):
        live = po.nplies > t
        if not bool(live.any()):
            break
        b, w = po.black[t][live].contiguous(), po.white[t][live].contiguous()
        own, opp = (b, w) if t % 2 == 0 else (w, b)
        legal = ops.legal(own, opp)
        two = (legal & (legal - 1)) != 0                                        # at least 2 bits set
        owns.append(own[two]); opps.append(opp[two])
    return torch.cat(owns).contiguous(), torch.cat(opps).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depths", default="1,2,4,6")
    ap.add_argument("--games", default="", help="games of the self-play run per depth, comma-separated")
    ap.add_argument("--lock-step", default="", help="games of the lock-step comparison per depth, comma-separated")
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_search_playout needs a CUDA device"
    dev = torch.device("cuda:0")
    depths = [int(x) for x in args.depths.split(",")]
    games = [int(x) for x in args.games.split(",")] if args.games else [GAMES[d] for d in depths]
    lock = [int(x) for x in args.lock_step.split(",")] if args.lock_step else [LOCK_STEP[d] for d in depths]
    w = torch.from_numpy(parameter.ProgressPositionMovesParameter().weights_table()).to(dev)
    for depth, n, n_lock in zip(depths, games, lock):
        info = gpu_info()
        play = lambda policy, out=None: ops.playout(n, seed=args.seed, device=dev, policy=policy, depth=depth,
                                                    random_plies=RANDOM_PLIES, weights=w, out=out)
        po = play(ops.POLICY_SEARCH)                                            # warm-up, same shape
        sec, po = events_time(lambda: play(ops.POLICY_SEARCH, po))
        plies = int(po.nplies.sum(dtype=torch.int64))
        own, opp = searched_positions(po, RANDOM_PLIES)
        _, _, nodes = ops.search(own, opp, w, depth, nodes=True)
        line = {"depth": depth, "games": n, "random_plies": RANDOM_PLIES, "kernel_s": round(sec, 4),
                "games_per_s": n / sec, "plies_per_s": plies / sec, "searched_positions": own.numel(),
                "searched_positions_per_s": own.numel() / sec, "nodes": int(nodes.sum()),
                "nodes_per_s": float(nodes.sum()) / sec, "nodes_per_searched_position": float(nodes.sum()) / own.numel()}
        if depth == 1:
            g = play(ops.POLICY_GREEDY)
            gsec, g = events_time(lambda: play(ops.POLICY_GREEDY, g))
            assert same_games(po, g), "depth-1 search self-play differs from the greedy kernel"
            line.update(greedy_kernel_s=round(gsec, 4), greedy_games_per_s=n / gsec)
        # the same kind of games without random plies, from 8-ply openings: the kernel against lock-step
        op = ops.playout(n_lock, seed=args.seed + 1, device=dev)
        b0, w0 = op.black[8].contiguous(), op.white[8].contiguous()
        kern = lambda m: ops.playout(m, device=dev, black0=b0[:m], white0=w0[:m], policy=ops.POLICY_SEARCH,
                                     depth=depth, weights=w)
        step = lambda m: play_search_games(m, w, depth, w, depth, dev, black0=b0[:m], white0=w0[:m])
        kern(64); step(64)                                                      # warm-up (both paths are loaded)
        ksec, k = wall_time(lambda: kern(n_lock))
        lsec, ls = wall_time(lambda: step(n_lock))
        assert same_games(k, ls), "the kernel's games differ from the lock-step games"
        line.update(lock_step_games=n_lock, from_ply=8, kernel_from_openings_s=round(ksec, 4),
                    lock_step_s=round(lsec, 4), lock_step_over_kernel=lsec / ksec, gpu=info)
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
