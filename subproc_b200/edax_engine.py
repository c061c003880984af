"""An engine process that speaks the text protocol ``game_runner.Player`` expects, backed by the GPU.

The reference plays a game by spawning two engines with ``subprocess.Popen(path, shell=True)`` and
talking to them over pipes (game_runner.py:11-102).  This module is such an engine:

    python -m subproc_b200.edax_engine [--policy random|greedy] [--param FILE] [--name NAME] [--seed S] [--exact N]
    python -m subproc_b200.edax_engine -h "<64 chars> <turn char>"      # feature dump

Protocol, as read by the reference's regexes:
  ``init``        -> 1 line (game_runner.py:35-39); resets to the standard opening
  ``go``          -> 3 lines which, joined, match ``>(.+) plays [WB]?([a-zA-Z][0-9]|PS)`` (:19-33);
                     the engine plays its own move
  ``<move>``      -> 3 lines matching ``(.+) play ([a-zA-Z][0-9]|PS|ps)`` (:41-54); the move is applied
  ``verbose p``   -> 1 line: the parameter set (:66-73);  ``verbose 0|1`` -> accepted
  ``quit``        -> 1 line, then exit (:56-64)
``-h "<sfen>"`` prints a Python list literal of the 9 features (mobility, a..h) of the colour named by
the turn character -- what parameter_learn_from_edax_protocol.counts parses (:7-13).  Which colour
the external engines meant is not pinned by the reference (the engines are not vendored).

``--exact N`` (default 0 = off): with at most N empty squares left, ``go`` plays the perfect-play move of the exact
endgame solver (ops.solve; the lowest square among the best moves) instead of the policy's.  N <= 24.

Move choice and all rules run through the CUDA kernels (subproc_b200.board / ops).
"""
import argparse
import sys


class Backend(object):
    """rules + policy on the GPU"""

    def __init__(self, policy='random', weights=None, seed=0, device=None, exact_empties=0):
        from . import board
        if exact_empties:
            from . import ops
            if not 0 < exact_empties <= ops.SOLVE_MAX_EMPTIES:
                raise ValueError("exact_empties must be in 0..%d" % ops.SOLVE_MAX_EMPTIES)
        self.board_mod = board
        self.policy = policy
        self.exact_empties = exact_empties
        self.weights = weights
        self.seed = seed
        self.device = device
        self.games = 0
        self.reset()

    def reset(self):
        self.b = self.board_mod.Board(device=self.device)
        self.games += 1

    def play(self, hand):
        return self.b.put_s(hand)

    def best_move(self):
        import numpy as np
        import torch
        from . import ops
        legal = self.b.puttables(self.b.turn)
        if not legal:
            return 'PS'
        own, opp = self.b._pair(self.b.turn)
        if 64 - bin(own | opp).count("1") <= self.exact_empties:
            dev = torch.device("cuda", self.b._ctx_index())
            _, move, _ = ops.solve(ops.bits_tensor([own], dev), ops.bits_tensor([opp], dev))
            s = int(move[0])
            return self.b.handstr_from_coord(s & 7, s >> 3).upper()
        if self.policy == 'random' or len(legal) == 1:
            key = (self.seed * 1000003 + self.games * 7919 + int(self.b.nturn)) & 0xFFFFFFFF
            x, y = legal[key % len(legal)] if self.policy == 'random' else legal[0]
            return self.b.handstr_from_coord(x, y).upper()
        dev = torch.device("cuda", self.b._ctx_index())
        n = len(legal)
        sq = torch.tensor([x + 8 * y for x, y in legal], dtype=torch.uint8, device=dev)
        o = ops.bits_tensor([own] * n, dev)
        p = ops.bits_tensor([opp] * n, dev)
        f = ops.flips(o, p, sq)
        o2 = o | f | ops.bits_tensor([1 << (x + 8 * y) for x, y in legal], dev)
        p2 = p & ~f
        side = torch.ones(n, dtype=torch.uint8, device=dev)            # evaluate (own', opp') as "Black" = own
        w = torch.from_numpy(np.asarray(self.weights, dtype=np.float32).reshape(4, 10)).to(dev)
        v = ops.evaluate(o2, p2, side, w).cpu().numpy()
        k = int(np.argmax(v))                                          # first maximum = lowest square
        return self.b.handstr_from_coord(*legal[k]).upper()

    def parameter_dump(self):
        return str(self.weights.tolist() if self.weights is not None else [])


class EdaxFrontEnd(object):
    """the line protocol; ``backend`` needs reset(), play(hand) -> int, best_move() -> str, parameter_dump()"""

    def __init__(self, backend, name='b200', out=None):
        self.backend = backend
        self.name = name
        self.out = out or sys.stdout

    def _say(self, *lines):
        for ln in lines:
            self.out.write(ln + "\n")
        self.out.flush()

    def handle(self, line):
        """returns False when the engine should exit"""
        cmd = line.strip()
        if cmd == 'init':
            self.backend.reset()
            self._say("init done")
        elif cmd == 'go':
            hand = self.backend.best_move()
            self.backend.play('ps' if hand.upper() == 'PS' else hand)
            self._say("", ">%s plays %s" % (self.name, hand), "")
        elif cmd == 'quit':
            self._say("bye")
            return False
        elif cmd.startswith('verbose'):
            arg = cmd.split()[1] if len(cmd.split()) > 1 else ''
            if arg == 'p':
                self._say(self.backend.parameter_dump())
            elif arg == '1':
                self._say(*([""] * 13))
            elif arg == '0':
                pass
        elif cmd:
            ret = self.backend.play(cmd)
            self._say("", "You play %s" % cmd if ret >= 0 else "You play %s (illegal)" % cmd, "")
        return True

    def serve(self, inp=None):
        inp = inp or sys.stdin
        for line in inp:
            if not self.handle(line):
                break


def feature_dump(sfen):
    """``-h "<64 chars> <turn>"`` -> list literal of 9 ints (parameter_learn_from_edax_protocol.py:7-13)"""
    from . import parameter
    book, turn = sfen[:64], (sfen[65] if len(sfen) > 65 else 'O')
    f = parameter.counts({'book': book, 'whosturn': turn, 'turn': 0}, turn)
    return str([int(v) for v in f[1:]])


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) >= 2 and argv[0] == '-h':
        print(feature_dump(argv[1]))
        return 0
    ap = argparse.ArgumentParser(add_help=False)
    ap.add_argument("--policy", default="greedy", choices=["random", "greedy"])
    ap.add_argument("--param", default=None, help="38-byte parameter file (paramgen format)")
    ap.add_argument("--name", default="b200")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--exact", type=int, default=0, help="play perfectly with at most this many empties (0 = off)")
    args = ap.parse_args(argv)
    from . import parameter, paramgen
    P = parameter.ProgressPositionMovesParameter()
    weights = P.weights_table(paramgen.read_data(args.param) if args.param else None)
    EdaxFrontEnd(Backend(args.policy, weights, args.seed, exact_empties=args.exact), args.name).serve()
    return 0


if __name__ == "__main__":
    sys.exit(main())
