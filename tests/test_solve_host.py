"""The exact endgame solver on the CPU: the reference solvers against each other, the host build of the search the
kernel runs (csrc/endgame.cuh) against them, hand-built positions that pin each rule of the semantics, and the
argument checks of othello_solve through the built library (no device needed)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import solve_util as su
from solve_util import BLACK, WHITE, PASS, NO_MOVE, REFUSED


def sample(oracle, empties, n, seed):
    parts = [su.positions_with_empties(oracle, e, n, seed + e) for e in empties]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def test_alphabeta_reference_equals_minimax(oracle):
    b, w, t = sample(oracle, range(0, 11), 30, 100)
    assert b.size > 250
    v0, m0 = su.oracle_solve(b, w, t, pruned=False)
    v1, m1 = su.oracle_solve(b, w, t, pruned=True)
    assert np.array_equal(v0, v1) and np.array_equal(m0, m1)


def test_host_search_equals_minimax_up_to_10_empties(oracle):
    b, w, t = sample(oracle, range(0, 11), 30, 200)
    v0, m0 = su.oracle_solve(b, w, t, pruned=False)
    v, m, nodes = su.host_solve(b, w, t)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)
    assert np.all(nodes >= 1)


def test_host_search_equals_alphabeta_at_12_to_14_empties(oracle):
    b, w, t = sample(oracle, (12,), 24, 300)
    b2, w2, t2 = su.positions_with_empties(oracle, 14, 4, 314)
    b, w, t = np.concatenate([b, b2]), np.concatenate([w, w2]), np.concatenate([t, t2])
    v0, m0 = su.oracle_solve(b, w, t, pruned=True)
    v, m, _ = su.host_solve(b, w, t)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)


@pytest.mark.parametrize("case", su.constructed_positions(), ids=lambda c: c[3])
def test_constructed_positions(case):
    b, w, turn, what = case
    v0, m0 = su.oracle_solve([b], [w], [turn], pruned=False)
    v, m, nodes = su.host_solve([b], [w], [turn])
    assert (v[0], m[0]) == (v0[0], m0[0]), what
    own, opp = (b, w) if turn == BLACK else (w, b)
    diff = bin(own).count("1") - bin(opp).count("1")
    if what.startswith("too many empties") or what == "overlap":
        assert (v[0], m[0], nodes[0]) == (REFUSED, NO_MOVE, 0)
    elif what.startswith("game over") or what.startswith("full board") or "nobody can move" in what:
        # the game is over: the disc difference as it stands, empties NOT given to the winner
        assert (v[0], m[0]) == (diff, NO_MOVE)
    elif what == "one empty, mover plays it":
        assert (v[0], m[0]) == (64, su.sq('h8'))
    elif what.startswith("one empty, mover must pass"):
        assert (v[0], m[0]) == (-64, PASS)
    elif what == "24 empties, root must pass":
        assert (v[0], m[0]) == (-41, PASS)
    elif what == "24 empties, three moves tie":
        assert (v[0], m[0]) == (41, su.sq('d6'))


def test_must_pass_and_game_over_roots(oracle):
    (pb, pw, pt), (ob, ow, ot) = su.special_positions(oracle, 40, 450, max_empties=10)
    assert pb.size >= 10 and ob.size == 40
    v0, m0 = su.oracle_solve(pb, pw, pt, pruned=False)
    v, m, _ = su.host_solve(pb, pw, pt)
    assert np.array_equal(v, v0) and np.array_equal(m, m0) and np.all(m == PASS)
    v_other, _, _ = su.host_solve(pb, pw, np.where(pt == BLACK, WHITE, BLACK))
    assert np.array_equal(v, -v_other)
    v, m, _ = su.host_solve(ob, ow, ot)
    own, opp = np.where(ot == BLACK, ob, ow), np.where(ot == BLACK, ow, ob)
    diff = np.array([bin(int(x)).count("1") - bin(int(y)).count("1") for x, y in zip(own, opp)])
    assert np.array_equal(v, diff) and np.all(m == NO_MOVE)


def test_root_pass_at_the_bound_on_empties():
    """A root with the most empties the solver accepts, whose mover must pass, is searched without a stack level
    beyond the bound: the host build with the bound lowered to 12 (and the register-resident levels to 2, so that the
    stack does nearly all the work) traps on a push past its last frame.  It runs in a child process so that a trap
    fails this test alone."""
    script = ("import sys; sys.path.insert(0, %r); import solve_util as su, numpy as np\n"
              "b, w = zip(*su.MUST_PASS_12)\n"
              "v, m, _ = su.host_solve(b, w, [su.BLACK] * len(b), defines=('OBE_MAX_EMPTIES=12', 'OBE_LOW_EMPTIES=2'))\n"
              "print(' '.join(map(str, v)), '|', ' '.join(map(str, m)))" % os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    vs, ms = r.stdout.strip().split("|")
    b, w = zip(*su.MUST_PASS_12)
    assert set(su.empties(b, w)) == {12}
    v0, m0 = su.oracle_solve(b, w, [BLACK] * len(b), pruned=True)
    assert [int(x) for x in vs.split()] == list(v0) and [int(x) for x in ms.split()] == list(m0)
    assert np.all(m0 == PASS)
    v, m, _ = su.host_solve(b, w, [BLACK] * len(b))                 # the product's setting
    assert np.array_equal(v, v0) and np.array_equal(m, m0)


def test_passes_inside_the_tree(oracle):
    b, w, t = su.positions_before_pass(oracle, 10, 60, 400)
    assert b.size >= 40
    v0, m0 = su.oracle_solve(b, w, t, pruned=False)
    v, m, _ = su.host_solve(b, w, t)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)


def test_ties_take_the_lowest_square(oracle):
    """positions where a higher square reaches the value too: the move is the lowest such square"""
    b, w, t = sample(oracle, range(2, 9), 25, 500)
    v, m, _ = su.host_solve(b, w, t)
    ties = 0
    for i in range(b.size):
        if m[i] >= 64:
            continue
        piece = int(t[i])
        legal = int(oracle.puttables([b[i]], [w[i]], piece)[0])
        squares = [s for s in range(64) if (legal >> s) & 1]
        cb, cw, _, _ = oracle.put(np.full(len(squares), b[i]), np.full(len(squares), w[i]), piece, squares)
        cv, _ = su.oracle_solve(cb, cw, np.full(len(squares), WHITE if piece == BLACK else BLACK), pruned=False)
        best = [s for s, c in zip(squares, cv) if -c == v[i]]
        assert m[i] == min(best)
        ties += len(best) > 1
    assert ties >= 20


def test_unreachable_bitboards():
    """arbitrary non-overlapping colourings with 6..10 empties, not reachable from the opening"""
    rng = np.random.RandomState(7)
    bs, ws, ts = [], [], []
    for i in range(100):
        empty = rng.choice(64, 6 + i % 5, replace=False)
        occ = ((1 << 64) - 1) & ~sum(1 << int(s) for s in empty)
        col = int(rng.randint(0, 2 ** 62, dtype=np.int64)) << 2 | int(rng.randint(0, 4))
        bs.append(occ & col); ws.append(occ & ~col); ts.append(BLACK if i % 2 else WHITE)
    b, w, t = np.array(bs, np.uint64), np.array(ws, np.uint64), np.array(ts, np.uint8)
    v0, m0 = su.oracle_solve(b, w, t, pruned=True)
    small = su.empties(b, w) <= 8
    v1, m1 = su.oracle_solve(b[small], w[small], t[small], pruned=False)
    assert np.array_equal(v0[small], v1) and np.array_equal(m0[small], m1)
    v, m, _ = su.host_solve(b, w, t)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)


def test_nodes_do_not_depend_on_the_batch(oracle):
    b, w, t = sample(oracle, (6, 9, 12), 20, 600)
    _, _, n0 = su.host_solve(b, w, t)
    p = np.random.RandomState(1).permutation(b.size)
    _, _, n1 = su.host_solve(b[p], w[p], t[p])
    assert np.array_equal(n1, n0[p])


def test_argument_validation_needs_no_gpu():
    from subproc_b200 import _lib
    L = _lib.lib()
    ws = L.othello_solve_workspace_bytes()
    assert ws > 0
    assert L.othello_solve(None, None, None, None, None, None, 0, None, 0, None) == 0          # n = 0: no-op
    assert L.othello_solve(None, None, None, None, None, None, 4, None, ws, None) == -1        # null pointers
    assert L.othello_solve(None, None, None, None, None, None, -1, None, ws, None) == -1       # n < 0
    buf = (ctypes.c_uint64 * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert L.othello_solve(p, p, None, p, p, None, 4, p, ws - 1, None) == -2                  # workspace too small
    assert L.othello_solve(p, p, None, p, None, None, 4, p, ws, None) == -1                   # move missing
