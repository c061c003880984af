#!/usr/bin/env python
"""tools/selfplay_learn.py -- the learning loop end to end on one GPU: greedy self-play with the
current integer weights -> on-GPU statistics -> refit -> +-127 scaling / int() -> next iteration,
then the learnt parameter set is matched against a random player and against the reference's
default_value() table (different engines per colour, both colour assignments).  Prints JSON lines.

    python tools/selfplay_learn.py [--depth D]

--depth D: the self-play games are search games at depth D (othello_playout, OTHELLO_POLICY_SEARCH) instead of greedy
ones; the lines carry "depth".  The greedy loop then runs too, with the same seeds and game ids, and a last line matches
the two learnt tables against each other, both played greedily."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from subproc_b200 import learner, parameter
from subproc_b200.game_runner import GameRunner, Engine

dev = "cuda:0"
P = parameter.ProgressPositionMovesParameter()
default = P.weights_table()


def match(a, b, n=32768, seed=100):
    """win rate of engine a against engine b over n games as Black + n games as White"""
    wins = games = 0
    for black, white, a_is_black in ((a, b, True), (b, a, False)):
        gr = GameRunner(black, white, None, False, 0, 0, device=dev, seed=seed)
        win = gr.winners(gr.play_games(n, trajectory=False)).cpu().numpy()
        wins += int((win == (1 if a_is_black else -1)).sum())
        games += n
        seed += 1
    return wins / games


ap = argparse.ArgumentParser()
ap.add_argument("--depth", type=int, default=None, help="search self-play at this depth (default: greedy self-play)")
args = ap.parse_args()
R = 6                                               # random opening plies in matches, for diversity
rand = Engine('random')


def learn(depth, report=True):
    L = learner.ProgressPositionMovesLearn()
    L.configure({})
    tag = {} if depth is None else {"depth": depth}
    if report:
        print(json.dumps(dict(tag, iteration=0, params=list(L.read_parameters()),
                              vs_random=match(Engine('greedy', default, random_plies=R), rand))), flush=True)
    t0 = time.perf_counter()
    for it in range(1, 13):
        po, rows = L.self_play_iteration(1 << 17, seed=7, iteration=it, random_plies=10, device=dev, depth=depth)
        if report and it % 4 == 0:
            learnt = Engine('greedy', L.weights_table(), random_plies=R)
            print(json.dumps(dict(tag, iteration=it, params=list(L.read_parameters()),
                                  r2=[round(f['r2'], 3) for f in L.last_fits],
                                  vs_random=match(learnt, rand),
                                  vs_default_value=match(learnt, Engine('greedy', default, random_plies=R)),
                                  elapsed_s=round(time.perf_counter() - t0, 2))), flush=True)
    return L


searched = learn(args.depth)
if args.depth is not None:
    greedy = learn(None, report=False)
    print(json.dumps({"depth": args.depth, "learnt_from_depth_vs_learnt_from_greedy": match(
        Engine('greedy', searched.weights_table(), random_plies=R), Engine('greedy', greedy.weights_table(), random_plies=R)),
        "greedy_learnt_params": list(greedy.read_parameters())}), flush=True)
