"""Helpers of the solver tests: the reference solver (tests/solve_oracle.c: negamax / alpha-beta on the oracle's
mailbox rules), the host build of the search the kernel runs (tests/solve_host.cpp -> csrc/endgame.cuh), and
positions with a given number of empty squares from seeded oracle playouts.

Both shared objects are built once per process (tests/host_build.py)."""
import ctypes
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

import host_build

BLACK, WHITE = 1, 2
PASS, NO_MOVE, REFUSED = 64, 255, -128

_solved = {}                                     # (black, white, turn, pruned) -> (value, move) of the reference


def oracle_lib():
    return host_build.load("solve_oracle.c")


def host_lib(defines=()):
    """the host build of csrc/endgame.cuh; defines (e.g. "OBE_MAX_EMPTIES=12") build a variant of the search"""
    return host_build.load("solve_host.cpp", defines)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _inputs(black, white, turn):
    b = np.ascontiguousarray(np.asarray(black, dtype=np.uint64).reshape(-1))
    w = np.ascontiguousarray(np.asarray(white, dtype=np.uint64).reshape(-1))
    t = np.full(b.size, BLACK, np.uint8) if turn is None else np.ascontiguousarray(np.asarray(turn, dtype=np.uint8).reshape(-1))
    return b, w, t


def oracle_solve(black, white, turn=None, pruned=False, threads=None):
    """(value int32[n], move uint8[n]) of orc_solve_ab (pruned) or orc_solve_minimax.  The positions are split over
    `threads` threads (ctypes releases the GIL), default one per core."""
    b, w, t = _inputs(black, white, turn)
    n = b.size
    value, move = np.zeros(n, np.int32), np.zeros(n, np.uint8)
    L = oracle_lib()
    key = lambda i: (int(b[i]), int(w[i]), int(t[i]), bool(pruned))

    def run(i):
        if key(i) not in _solved:
            L.orc_solve_batch(_p(b[i:]), _p(w[i:]), _p(t[i:]), ctypes.c_int(1 if pruned else 0), _p(value[i:]),
                              _p(move[i:]), ctypes.c_int64(1))
            _solved[key(i)] = (value[i], move[i])
        value[i], move[i] = _solved[key(i)]

    with ThreadPoolExecutor(threads or os.cpu_count() or 1) as ex:
        list(ex.map(run, range(n)))
    return value, move


def host_solve(black, white, turn=None, defines=()):
    """(value, move, nodes) of the host build of csrc/endgame.cuh, one core"""
    b, w, t = _inputs(black, white, turn)
    n = b.size
    value, move, nodes = np.zeros(n, np.int32), np.zeros(n, np.uint8), np.zeros(n, np.uint64)
    host_lib(defines).eg_solve(_p(b), _p(w), _p(t), _p(value), _p(move), _p(nodes), ctypes.c_long(n))
    return value, move, nodes


def empties(black, white):
    occ = np.asarray(black, dtype=np.uint64) | np.asarray(white, dtype=np.uint64)
    return np.array([64 - bin(int(v)).count("1") for v in occ], dtype=np.int32)


def positions_with_empties(oracle, n_empties, n, seed, games=None):
    """Up to n positions (black, white, turn) with exactly n_empties empty squares, the first such position of each
    of the seeded oracle random playouts (the side to move alternates every ply, passes included)."""
    games = games or 2 * n
    r = oracle.playout(seed, 0, games)
    bs, ws, ts = [], [], []
    for g in range(games):
        for t in range(int(r['nplies'][g]) + 1):
            b, w = int(r['black'][t, g]), int(r['white'][t, g])
            if 64 - bin(b | w).count("1") == n_empties:
                bs.append(b); ws.append(w); ts.append(BLACK if t % 2 == 0 else WHITE)
                break
        if len(bs) == n:
            break
    return np.array(bs, np.uint64), np.array(ws, np.uint64), np.array(ts, np.uint8)


def special_positions(oracle, n, seed, max_empties=64):
    """Must-pass and game-over roots (at most max_empties empties) from seeded oracle playouts: (black, white, turn)
    of each kind."""
    games = 40 * n
    r = oracle.playout(seed, 0, games)
    pb, pw, pt, ob, ow, ot = [], [], [], [], [], []
    few = lambda b, w: 64 - bin(int(b) | int(w)).count("1") <= max_empties
    for g in range(games):
        L = int(r['nplies'][g])
        if len(ob) < n and few(r['final_black'][g], r['final_white'][g]):
            ob.append(int(r['final_black'][g])); ow.append(int(r['final_white'][g])); ot.append(BLACK if L % 2 == 0 else WHITE)
        for t in range(L):
            if r['move'][t, g] == PASS and len(pb) < n and few(r['black'][t, g], r['white'][t, g]):
                pb.append(int(r['black'][t, g])); pw.append(int(r['white'][t, g])); pt.append(BLACK if t % 2 == 0 else WHITE)
    as_arrays = lambda b, w, t: (np.array(b, np.uint64), np.array(w, np.uint64), np.array(t, np.uint8))
    return as_arrays(pb, pw, pt), as_arrays(ob, ow, ot)


def sq(name):
    """'a1' -> 0, 'h8' -> 63"""
    return (ord(name[0]) - ord('a')) + 8 * (int(name[1]) - 1)


def bits(*names):
    v = 0
    for s in names:
        v |= 1 << sq(s)
    return v


def constructed_positions():
    """Hand-built positions, each pinning one rule: (black, white, turn, what)."""
    full = (1 << 64) - 1
    cases = []
    # a full board: game over, value = disc difference, no move
    b = 0x00000000FFFFFFFF
    cases.append((b, full & ~b, BLACK, "full board"))
    # game over with empty squares left (a8, h1): every line through them is Black up to the edge, White's one disc
    # (d4) is on none of them; the value is the disc difference, the empties are not given to the winner
    b = full & ~bits('a8', 'h1', 'd4')
    cases.append((b, bits('d4'), BLACK, "game over, empties left"))
    cases.append((b, bits('d4'), WHITE, "game over, empties left, White to move"))
    # one empty square (h8), Black to move can take it
    w = bits('g8', 'g7', 'h7')
    b = full & ~w & ~bits('h8')
    cases.append((b, w, BLACK, "one empty, mover plays it"))
    cases.append((b, w, WHITE, "one empty, mover must pass, opponent plays it"))
    # one empty (h8) that nobody can take: every line through it is Black up to the edge, the one White disc is on none
    b = full & ~bits('h8', 'b3')
    cases.append((b, bits('b3'), BLACK, "one empty, nobody can move"))
    cases.append((b, bits('b3'), WHITE, "one empty, nobody can move, White to move"))
    # exactly 24 empties (ranks 6-8), White's one disc e5 among Black's ranks 1-5: White must pass; Black's d6, e6 and f6
    # each flip e5 and end the game (a tie between three squares at the root of the other side)
    b = ((1 << 40) - 1) & ~bits('e5')
    cases.append((b, bits('e5'), WHITE, "24 empties, root must pass"))
    cases.append((b, bits('e5'), BLACK, "24 empties, three moves tie"))
    # refused: 25 empties (the same without a1), the start position (60 empties) and overlapping colours
    cases.append((b & ~bits('a1'), bits('e5'), BLACK, "too many empties: 25"))
    cases.append((0x0000000810000000, 0x0000001008000000, BLACK, "too many empties"))
    cases.append((bits('a1', 'b1'), bits('b1', 'c1'), BLACK, "overlap"))
    return cases


def positions_before_pass(oracle, max_empties, n, seed):
    """Up to n positions with at most max_empties empties whose game goes on to a pass: the line played is a path of
    the search tree, so the tree has a pass inside."""
    games = 8 * n
    r = oracle.playout(seed, 0, games)
    bs, ws, ts = [], [], []
    for g in range(games):
        L = int(r['nplies'][g])
        passes = [t for t in range(L) if r['move'][t, g] == PASS]
        for t in range(L):
            b, w = int(r['black'][t, g]), int(r['white'][t, g])
            if 64 - bin(b | w).count("1") <= max_empties and any(p > t for p in passes):
                bs.append(b); ws.append(w); ts.append(BLACK if t % 2 == 0 else WHITE)
                break
        if len(bs) == n:
            break
    return np.array(bs, np.uint64), np.array(ws, np.uint64), np.array(ts, np.uint8)


# Roots with 12 empties whose mover (Black) must pass, arbitrary colourings found by rejection sampling: with
# OBE_MAX_EMPTIES=12 the host build searches them at the bound on empties, down its whole stack.
MUST_PASS_12 = [
    (0x4199dbdef96f5821, 0xbe0604010600818c), (0xd2a01d52372c8e2d, 0x2d0f828d888070d0),
    (0x0098326c3f4f371d, 0x5f070d93c08000e0), (0x8c4ced0a537d264d, 0x73b300818080c1b2),
    (0x0b54ca9a7eaf5f80, 0xf42831608040a023), (0x2868aedd37b02f0c, 0x871741008043d0f0),
    (0x28c0e9bfc86cfac5, 0x811900403713013a), (0xd12434bbe8fa8a65, 0x0e99c90003052198),
    (0x3cb0fdbab535352d, 0xc0400005428a82d2), (0x183d5fcc33163a9a, 0x87822031c0e0c160),
    (0x03fa1dcc2cebf873, 0x4801e033d110000c), (0x023e567d747cee25, 0x418181820b031198)]
