"""The reference's GameRunner (game_runner.py:105-201) over the lock-step playout kernel.

The reference plays ONE game between two engine subprocesses; here the "engines" are policies
evaluated inside the playout kernels, and ``play_games(n)`` plays n games in one launch.  The
constructor keeps the reference's argument order (game_runner.py:107): where the reference takes
two shell commands, this takes two engine specs -- Black's and White's may differ (random vs greedy,
or two greedy engines with different parameter sets), like proc_black / proc_white.

The recorder protocol is the reference's: ``recorder.add(board)`` for the initial position and
after every ply (game_runner.py:170,159), ``add_meta`` + ``store`` at the end (:186-192).  Boards
handed to recorders are ``subproc_b200.board.Board`` objects rebuilt from the trajectory.

A 'search' engine (depth-limited alpha-beta on a weight table, ops.search) is not inside the playout kernels: when
either side is one, the games are played in lock-step from the host (``play_search_games``), one search launch per
colour and one step launch per ply, into the same ``ops.Playout`` the kernels fill.
"""
import torch

from . import ops
from . import board as board_mod

N_RAND_HAND_UNTIL = 10                               # game_runner.py:6 (applied inside the kernel)


class Engine(object):
    """What sits behind Player.go (game_runner.py:19-33): 'random', 'greedy' on a weight table, or 'search' -- the
    minimax move of a ``depth``-ply alpha-beta search on a weight table (depth 1 is 'greedy')."""

    def __init__(self, policy='random', weights=None, random_plies=0, name=None, depth=None):
        if policy not in ('random', 'greedy', 'search'):
            raise ValueError("engine policy must be 'random', 'greedy' or 'search'")
        if policy == 'search' and not (depth is not None and 1 <= int(depth) <= ops.SEARCH_MAX_DEPTH):
            raise ValueError("a search engine needs depth in 1..%d" % ops.SEARCH_MAX_DEPTH)
        self.policy = policy
        self.weights = weights                       # 4 x 9 (default_value() layout) or 4 x 10
        self.random_plies = random_plies
        self.depth = int(depth) if policy == 'search' else (1 if policy == 'greedy' else None)
        self.name = name or ('b200-' + policy + ('%d' % self.depth if policy == 'search' else ''))


def play_search_games(n_games, weights_black, depth_black, weights_white, depth_white, device, black0=None, white0=None,
                      turn0=None, trajectory=True, t_max=ops.T_MAX_DEFAULT, out=None):
    """n_games games in lock-step between two search engines (float32 [4][10] device tables, depths 1..12; a greedy
    engine is depth 1), from the standard opening or from black0 / white0 (int64 [n]) with turn0 (uint8 [n], None =
    Black) to move.  Every ply is one ops.search launch per colour that has live games, then one ops.step; the host
    synchronises once per ply, to learn how many games each colour has to move.  Returns an ops.Playout like
    ops.playout: trajectory rows, nplies, final positions (rows past a game's end hold its final position)."""
    device = torch.device(device)
    n = int(n_games)
    full = lambda v, dtype: torch.full((n,), v, dtype=dtype, device=device)
    b = full(ops.signed64(ops.START_BLACK), torch.int64) if black0 is None else black0.clone()
    w = full(ops.signed64(ops.START_WHITE), torch.int64) if white0 is None else white0.clone()
    turn = full(ops.BLACK, torch.uint8) if turn0 is None else turn0.clone()
    nturn = full(0, torch.int32)
    if out is None:
        tb = torch.empty((t_max + 1, n), dtype=torch.int64, device=device) if trajectory else None
        tw = torch.empty((t_max + 1, n), dtype=torch.int64, device=device) if trajectory else None
        tm = torch.empty((t_max, n), dtype=torch.uint8, device=device) if trajectory else None
        out = ops.Playout(n, t_max, tb, tw, tm, torch.empty(n, dtype=torch.int32, device=device),
                          torch.empty(n, dtype=torch.int64, device=device), torch.empty(n, dtype=torch.int64, device=device))
    live = (ops.legal(b, w) | ops.legal(w, b)) != 0
    engines = ((ops.BLACK, weights_black, depth_black), (ops.WHITE, weights_white, depth_white))
    move = full(ops.NO_MOVE, torch.uint8)
    t = 0
    while True:
        to_move = [live & (turn == c) for c, _, _ in engines]
        counts = torch.stack([m.sum() for m in to_move]).tolist()         # the one synchronisation of the ply
        if sum(counts) == 0:
            break
        if out.black is not None and t <= out.t_max:
            out.black[t].copy_(b)
            out.white[t].copy_(w)
        move.fill_(ops.NO_MOVE)                                            # finished games: no move, state untouched
        for (c, weights, depth), mask, k in zip(engines, to_move, counts):
            if k == 0:
                continue
            idx = torch.argsort(mask.to(torch.int32), descending=True, stable=True)[:k]
            _, mv, _ = ops.search(b[idx], w[idx], weights, depth, turn=turn[idx])
            move[idx] = mv
        if out.move is not None and t < out.t_max:
            out.move[t].copy_(move)
        _, _, flags = ops.step(b, w, turn, nturn, move)
        live &= (flags & ops.F_GAME_OVER) == 0
        t += 1
    if out.black is not None and t <= out.t_max:
        out.black[t:].copy_(b.expand(out.t_max + 1 - t, n))
        out.white[t:].copy_(w.expand(out.t_max + 1 - t, n))
    out.nplies.copy_(nturn)
    out.final_black.copy_(b)
    out.final_white.copy_(w)
    return out


class GameRunner(object):
    def __init__(self, proc_black, proc_white, game_recorder=None, debug=False, n_rand_hands_for_black=0,
                 n_rand_hands_for_white=0, device=None, seed=0):
        if not isinstance(proc_black, Engine):
            proc_black = Engine(proc_black)
        if not isinstance(proc_white, Engine):
            proc_white = Engine(proc_white)
        self.proc_black, self.proc_white = proc_black, proc_white
        self.recorder = game_recorder
        self.debug = debug
        self.n_rand_black = int(n_rand_hands_for_black)
        self.n_rand_white = int(n_rand_hands_for_white)
        self.device = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
        self.seed = seed
        self.next_gid = 0
        greedy = [e for e in (proc_black, proc_white) if e.policy == 'greedy']
        if len(greedy) == 2 and greedy[0].random_plies != greedy[1].random_plies:
            raise ValueError("the two greedy engines must share random_plies (one opening length per game)")
        self.random_plies = greedy[0].random_plies if greedy else 0
        self.lock_step = any(e.policy == 'search' for e in (proc_black, proc_white))
        if self.lock_step and ('random' in (proc_black.policy, proc_white.policy) or self.random_plies > 0 or
                               self.n_rand_black > 0 or self.n_rand_white > 0):
            raise ValueError("a search engine plays against a search or greedy engine, without random plies or "
                             "random-hand substitution")
        self._weights = [self._table(e) for e in (proc_black, proc_white)]

    def _table(self, engine):
        if engine.policy == 'random':
            return None
        import numpy as np
        w = np.asarray(engine.weights, dtype=np.float64).reshape(4, -1)
        return ops.weights_tensor(w[:, :9], self.device, w[:, 9] if w.shape[1] > 9 else None)

    def play_games(self, n_games, trajectory=True, t_max=ops.T_MAX_DEFAULT, out=None):
        """n_games games in one launch (in lock-step from the host when a side is a search engine); returns an
        ops.Playout (trajectories stay in HBM)."""
        if self.lock_step:
            po = play_search_games(n_games, self._weights[0], self.proc_black.depth, self._weights[1],
                                   self.proc_white.depth, self.device, trajectory=trajectory, t_max=t_max, out=out)
            self.next_gid += int(n_games)
            return po
        pol = [ops.POLICY_GREEDY if e.policy == 'greedy' else ops.POLICY_RANDOM for e in (self.proc_black, self.proc_white)]
        po = ops.playout(n_games, seed=self.seed, gid0=self.next_gid, device=self.device, policy=pol[0],
                         policy_white=pol[1], random_plies=self.random_plies, n_rand_black=self.n_rand_black,
                         n_rand_white=self.n_rand_white, weights=self._weights[0], weights_white=self._weights[1],
                         t_max=t_max, trajectory=trajectory, out=out)
        self.next_gid += int(n_games)
        return po

    def winners(self, po):
        """int8[n]: +1 Black won, -1 White won, 0 draw (game_runner.py:194-199)."""
        c = po.final_counts()
        return torch.sign(c[:, 0] - c[:, 1]).to(torch.int8)

    def play_a_game(self):
        """One game with the reference's return value ((colour, engine name)) and recorder calls."""
        po = self.play_games(1)
        n = int(po.nplies.cpu()[0])
        if self.recorder is not None:
            blacks = ops.bits_numpy(po.black[:n + 1, 0])
            whites = ops.bits_numpy(po.white[:n + 1, 0])
            turn = board_mod.Black
            for t in range(n + 1):
                b = board_mod.Board(device=self.device)
                b._black, b._white, b.turn, b.nturn = int(blacks[t]), int(whites[t]), turn, t
                self.recorder.add(b)
                turn = b.hostile(turn)
            self.recorder.add_meta({'proc_a': self.proc_black.name, 'proc_b': self.proc_white.name,
                                    'hamletparam': 'No Hamlet'})
            self.recorder.store()
        c = po.final_counts().cpu()
        nb, nw = int(c[0, 0]), int(c[0, 1])
        if nb > nw:
            return ("Black", self.proc_black.name)
        if nb < nw:
            return ("White", self.proc_white.name)
        return ("None", '')
