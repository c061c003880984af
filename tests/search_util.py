"""Helpers of the midgame search tests: the reference search (tests/search_oracle.c: plain minimax / unordered
alpha-beta on the oracle's mailbox rules and fp64 evaluation), the host build of the search the kernel runs
(tests/search_host.cpp -> csrc/midgame.cuh), weight tables and sampled positions.

Both shared objects are built once per process into a temporary directory."""
import ctypes
import os
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np

import solve_util as su

HERE = os.path.dirname(os.path.abspath(__file__))
BLACK, WHITE, PASS, NO_MOVE = su.BLACK, su.WHITE, su.PASS, su.NO_MOVE
MAX_DEPTH = 12

_libs = {}


def _build(name, cmd):
    if name not in _libs:
        out = os.path.join(tempfile.mkdtemp(prefix="search_"), name + ".so")
        subprocess.check_call(cmd + ["-o", out])
        _libs[name] = ctypes.CDLL(out)
    return _libs[name]


def oracle_lib():
    return _build("search_oracle", ["gcc", "-O2", "-std=c99", "-shared", "-fPIC", os.path.join(HERE, "search_oracle.c"),
                                    "-lm"])


def host_lib():
    """the host build of csrc/midgame.cuh; -std=c++17 so that g++ contracts no float expression"""
    L = _build("search_host", ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++",
                               os.path.join(HERE, "search_host.cpp")])
    L.mg_score.restype = ctypes.c_float
    L.mg_score.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def weights40(w):
    return np.ascontiguousarray(np.asarray(w, dtype=np.float32).reshape(4, 10))


def default_weights():
    from oracle import lib as orc
    return weights40(orc.DEFAULT_WEIGHTS)


def int_weights(seed):
    """a random integer table in -127..127, intercepts included"""
    return weights40(np.random.RandomState(seed).randint(-127, 128, size=(4, 10)))


def float_weights(seed):
    """a random three-decimal table with intercepts: scores are not integers, sums round"""
    return weights40(np.round(np.random.RandomState(seed).uniform(-20, 20, size=(4, 10)), 3))


def _inputs(black, white, turn):
    b = np.ascontiguousarray(np.asarray(black, dtype=np.uint64).reshape(-1))
    w = np.ascontiguousarray(np.asarray(white, dtype=np.uint64).reshape(-1))
    t = np.full(b.size, BLACK, np.uint8) if turn is None else np.ascontiguousarray(np.asarray(turn, dtype=np.uint8).reshape(-1))
    return b, w, t


def oracle_search(black, white, turn, weights, depth, pruned=False, threads=None):
    """(value float64 [n], move uint8 [n]) of the reference, positions split over threads (ctypes releases the GIL)"""
    b, w, t = _inputs(black, white, turn)
    n = b.size
    value, move = np.zeros(n, np.float64), np.zeros(n, np.uint8)
    wd = np.ascontiguousarray(weights40(weights).astype(np.float64))
    L = oracle_lib()

    def run(i):
        L.orc_search_batch(_p(b[i:]), _p(w[i:]), _p(t[i:]), _p(wd), ctypes.c_int(depth), ctypes.c_int(1 if pruned else 0),
                           _p(value[i:]), _p(move[i:]), ctypes.c_int64(1))

    with ThreadPoolExecutor(threads or os.cpu_count() or 1) as ex:
        list(ex.map(run, range(n)))
    return value, move


def oracle_children(black, white, turn, weights, depth):
    """float64 [64]: the minimax value of each root move's subtree from the root mover's side, NaN where illegal"""
    out = np.zeros(64, np.float64)
    wd = np.ascontiguousarray(weights40(weights).astype(np.float64))
    oracle_lib().orc_search_children(ctypes.c_uint64(int(black)), ctypes.c_uint64(int(white)), ctypes.c_int(int(turn)),
                                     _p(wd), ctypes.c_int(depth), _p(out))
    return out


def positions_pass_after(oracle, k, n, seed):
    """Up to n positions from seeded oracle random playouts whose game passes exactly k plies later: searched to depth
    k + 1, the line played has its pass on the last ply."""
    games = 40 * n
    r = oracle.playout(seed, 0, games)
    bs, ws, ts = [], [], []
    for g in range(games):
        L = int(r['nplies'][g])
        for t in range(L - k):
            if r['move'][t + k, g] == PASS and (k == 0 or r['move'][t, g] != PASS):
                bs.append(int(r['black'][t, g])); ws.append(int(r['white'][t, g])); ts.append(BLACK if t % 2 == 0 else WHITE)
                break
        if len(bs) == n:
            break
    return np.array(bs, np.uint64), np.array(ws, np.uint64), np.array(ts, np.uint8)


def positions_before_end(oracle, k, n, seed):
    """Up to n positions k plies before the end of their seeded oracle random playout (game over inside a tree of
    depth > k)"""
    r = oracle.playout(seed, 0, n)
    t = r['nplies'].astype(np.int64) - k
    g = np.nonzero(t >= 0)[0]
    b, w = r['black'][t[g], g], r['white'][t[g], g]
    return b.astype(np.uint64), w.astype(np.uint64), np.where(t[g] % 2 == 0, BLACK, WHITE).astype(np.uint8)


def host_search(black, white, turn, weights, depth):
    """(value float32, move uint8, nodes uint64) of the host build of csrc/midgame.cuh, one core"""
    b, w, t = _inputs(black, white, turn)
    n = b.size
    value, move, nodes = np.zeros(n, np.float32), np.zeros(n, np.uint8), np.zeros(n, np.uint64)
    wf = weights40(weights)
    host_lib().mg_search(_p(b), _p(w), _p(t), _p(wf), ctypes.c_int(depth), _p(value), _p(move), _p(nodes),
                         ctypes.c_long(n))
    return value, move, nodes


def host_score(P, O, weights):
    wf = weights40(weights)
    L = host_lib()
    return np.array([L.mg_score(int(p), int(o), _p(wf)) for p, o in zip(P, O)], np.float32)


def spread(oracle, per_empties, seed, lo=0, hi=56):
    """positions from lo..hi empties (per_empties of each, first of each seeded oracle random playout), plus must-pass
    and game-over roots: (black, white, turn)"""
    parts = [su.positions_with_empties(oracle, e, per_empties, seed + e) for e in range(lo, hi + 1)]
    (pb, pw, pt), (ob, ow, ot) = su.special_positions(oracle, max(2, per_empties), seed + 99)
    parts += [(pb, pw, pt), (ob, ow, ot)]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def successors(oracle, b, w, turn):
    """the legal moves of the side to move and the positions after them: (squares, black', white')"""
    legal = int(oracle.puttables([b], [w], turn)[0])
    squares = [s for s in range(64) if (legal >> s) & 1]
    cb, cw, _, _ = oracle.put(np.full(len(squares), b, np.uint64), np.full(len(squares), w, np.uint64), turn, squares)
    return squares, cb, cw
