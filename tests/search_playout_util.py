"""The referee of the search self-play tests: GameRunner.play_a_game on the host, with the oracle's rules and RNG and
the reference search (or the host build of csrc/midgame.cuh) behind a search engine.

Every game is played from scratch by the rules othello_playout documents for OTHELLO_POLICY_SEARCH: the draws
rng_draw(key, t, 0) (substitution, budget min(n_rand, 10)) and rng_draw(key, t, 1) (the random move, the k-th legal
square with k = below(r, n) = (r * n) >> 32), random plies while t < random_plies, no search for a forced move or a
pass.  The games of a batch advance one ply at a time, so the searches of a ply go to the reference in one batch."""
import numpy as np

import search_util as xu

BLACK, WHITE, PASS = xu.BLACK, xu.WHITE, xu.PASS
RANDOM, GREEDY, SEARCH = 0, 1, 2


def below(r, n):
    return (int(r) * int(n)) >> 32


def kth_square(mask, k):
    for s in range(64):
        if (mask >> s) & 1:
            if k == 0:
                return s
            k -= 1
    raise ValueError("k-th square of a mask with fewer squares")


def oracle_searcher(black, white, turn, weights, depth):
    """the reference search's moves (plain minimax up to depth 3, alpha-beta above): integer weights only"""
    return xu.oracle_search(black, white, turn, weights, depth, pruned=depth > 3)[1]


def host_searcher(black, white, turn, weights, depth):
    """the moves of the host build of the search the kernel runs: bit-exact for float weights"""
    return xu.host_search(black, white, turn, weights, depth)[1]


def referee(oracle, n, seed=0, gid0=0, black0=None, white0=None, turn0=None, policy=SEARCH, policy_white=None,
            depth=1, depth_white=None, random_plies=0, n_rand_black=0, n_rand_white=0, weights=None,
            weights_white=None, t_max=120, searcher=oracle_searcher):
    """n games gid0.. : dict(black [t_max+1][n], white, move [t_max][n], nplies, final_black, final_white, totals,
    searched) -- trajectory entries past a game's end are 0 (moves 255); `searched` lists (black, white, colour)
    of every ply that went to the search"""
    policy_white = policy if policy_white is None else policy_white
    depth_white = depth if depth_white is None else depth_white
    weights_white = weights if weights_white is None else weights_white
    engine = {BLACK: (policy, depth, weights), WHITE: (policy_white, depth_white, weights_white)}
    # a greedy engine is a search engine of depth 1
    engine = {c: (0 if p == RANDOM else (1 if p == GREEDY else d), w) for c, (p, d, w) in engine.items()}
    b = np.full(n, 0x0000000810000000, np.uint64) if black0 is None else np.asarray(black0, np.uint64).copy()
    w = np.full(n, 0x0000001008000000, np.uint64) if white0 is None else np.asarray(white0, np.uint64).copy()
    turn = np.full(n, BLACK, np.uint8) if turn0 is None else np.where(np.asarray(turn0) == BLACK, BLACK, WHITE).astype(np.uint8)
    keys = [oracle.rng_key(seed, gid0 + g) for g in range(n)]
    rest = {BLACK: [min(n_rand_black, 10)] * n, WHITE: [min(n_rand_white, 10)] * n}
    tb, tw = np.zeros((t_max + 1, n), np.uint64), np.zeros((t_max + 1, n), np.uint64)
    mv = np.full((t_max, n), 255, np.uint8)
    nplies = np.zeros(n, np.int32)
    tb[0], tw[0] = b, w
    live = oracle.game_over(b, w) == 0
    searched = []
    t = 0
    while live.any():
        legal = np.where(turn == BLACK, oracle.puttables(b, w, BLACK), oracle.puttables(b, w, WHITE))
        move = np.full(n, PASS, np.uint8)
        ask = {BLACK: [], WHITE: []}                              # games whose engine searches this ply
        for g in np.nonzero(live)[0]:
            m = int(legal[g])
            if m == 0:
                continue
            c = int(turn[g])
            cnt = bin(m).count("1")
            d = engine[c][0]
            random_now = t < random_plies or d == 0
            if rest[c][g] > 0 and below(oracle.rng_draw(keys[g], t, 0), rest[c][g]) == 0:
                random_now = True
                rest[c][g] -= 1
            if random_now:
                move[g] = kth_square(m, below(oracle.rng_draw(keys[g], t, 1), cnt))
            elif cnt == 1:
                move[g] = kth_square(m, 0)
            else:
                ask[c].append(g)
        for c, games in ask.items():
            if games:
                idx = np.array(games)
                d, wt = engine[c]
                move[idx] = searcher(b[idx], w[idx], turn[idx], wt, d)
                searched += [(int(b[g]), int(w[g]), c) for g in games]
        if t < t_max:
            mv[t, live] = move[live]
        idx = np.nonzero(live)[0]
        nb, nw, nt, _, _, _ = oracle.step(b[idx], w[idx], turn[idx], np.full(idx.size, t), move[idx])
        b[idx], w[idx], turn[idx] = nb, nw, nt
        t += 1
        nplies[idx] = t
        if t <= t_max:
            tb[t, idx], tw[t, idx] = nb, nw
        live[idx] = oracle.game_over(b[idx], w[idx]) == 0
    c = oracle.counts(b, w).astype(np.int64)
    totals = np.array([int(nplies.sum()), int((c[:, 0] - c[:, 1]).sum()), int((c[:, 0] > c[:, 1]).sum()),
                       int((c[:, 1] > c[:, 0]).sum())], np.int64)
    return dict(black=tb, white=tw, move=mv, nplies=nplies, final_black=b, final_white=w, totals=totals,
                searched=searched)
