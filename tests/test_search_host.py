"""The midgame search on the CPU: the host build of the search the kernel runs (csrc/midgame.cuh) against the
reference minimax / alpha-beta of tests/search_oracle.c with integer weights (every score an exact integer, so the
comparison is ==), hand-built and sampled positions that pin each rule of the semantics, and the argument checks of
othello_search through the built library (no device needed)."""
import ctypes

import numpy as np
import pytest

import search_util as xu
import solve_util as su
from search_util import BLACK, WHITE, PASS, NO_MOVE

TABLES = {"default": xu.default_weights, "int7": lambda: xu.int_weights(7), "int8": lambda: xu.int_weights(8)}


def check_against_oracle(b, w, t, weights, depth, pruned):
    v0, m0 = xu.oracle_search(b, w, t, weights, depth, pruned=pruned)
    v, m, nodes = xu.host_search(b, w, t, weights, depth)
    assert np.array_equal(v.astype(np.float64), v0), depth
    assert np.array_equal(m, m0), depth
    assert np.all(nodes >= 1)
    return v, m, nodes


@pytest.fixture(scope="module")
def spread(oracle):
    return xu.spread(oracle, 5, 100)


@pytest.mark.parametrize("table", sorted(TABLES))
@pytest.mark.parametrize("depth", [1, 2, 3])
def test_host_equals_minimax(spread, table, depth):
    b, w, t = spread
    assert b.size > 280
    check_against_oracle(b, w, t, TABLES[table](), depth, pruned=False)


def test_alphabeta_reference_equals_minimax(spread):
    b, w, t = (a[::3] for a in spread)
    weights = xu.int_weights(3)
    assert [np.array_equal(x, y) for x, y in zip(xu.oracle_search(b, w, t, weights, 3, pruned=False),
                                                 xu.oracle_search(b, w, t, weights, 3, pruned=True))] == [True, True]


@pytest.mark.parametrize("table", ["default", "int7"])
@pytest.mark.parametrize("depth", [4, 5])
def test_host_equals_alphabeta(spread, table, depth):
    b, w, t = (a[::4] for a in spread)
    check_against_oracle(b, w, t, TABLES[table](), depth, pruned=True)


def test_root_must_pass(oracle):
    b, w = (np.array(a, np.uint64) for a in zip(*su.MUST_PASS_12))
    (pb, pw, pt), _ = su.special_positions(oracle, 20, 450)
    b, w, t = np.concatenate([b, pb]), np.concatenate([w, pw]), np.concatenate([np.full(b.size, BLACK, np.uint8), pt])
    weights = xu.int_weights(11)
    for depth in (1, 2, 3, 4):
        v, m, _ = check_against_oracle(b, w, t, weights, depth, pruned=True)
        assert np.all(m == PASS)
    # depth 1: the passed position is a leaf, scored from the root mover's side
    v, _, nodes = xu.host_search(b, w, t, weights, 1)
    own, opp = np.where(t == BLACK, b, w), np.where(t == BLACK, w, b)
    assert np.array_equal(v, xu.host_score(own, opp, weights)) and np.all(nodes == 2)


@pytest.mark.parametrize("k", [0, 1, 2])
def test_pass_inside_the_tree_at_the_last_level(oracle, k):
    b, w, t = xu.positions_pass_after(oracle, k, 40, 700 + k)
    assert b.size >= 20
    for depth in (k + 1, k + 2):
        check_against_oracle(b, w, t, xu.int_weights(k), depth, pruned=False)


def test_game_over_at_the_root_and_inside_the_tree(oracle):
    weights = xu.int_weights(5)
    _, (ob, ow, ot) = su.special_positions(oracle, 30, 800)
    v, m, nodes = check_against_oracle(ob, ow, ot, weights, 3, pruned=False)
    own, opp = np.where(ot == BLACK, ob, ow), np.where(ot == BLACK, ow, ob)
    assert np.all(m == NO_MOVE) and np.all(nodes == 1)
    assert np.array_equal(v, xu.host_score(own, opp, weights))
    for k in (1, 2, 3):
        b, w, t = xu.positions_before_end(oracle, k, 60, 810 + k)
        check_against_oracle(b, w, t, weights, k + 2, pruned=k >= 3)


def test_full_board_and_overlap():
    full = (1 << 64) - 1
    weights = xu.int_weights(9)
    b = np.array([0x00000000FFFFFFFF, 0x00000000FFFFFFFF, 3], np.uint64)
    w = np.array([full & ~0x00000000FFFFFFFF, full & ~0x00000000FFFFFFFF, 6], np.uint64)
    t = np.array([BLACK, WHITE, BLACK], np.uint8)
    for depth in (1, 6, 12):
        v, m, nodes = xu.host_search(b, w, t, weights, depth)
        assert v[0] == xu.host_score(b[:1], w[:1], weights)[0] and v[1] == xu.host_score(w[1:2], b[1:2], weights)[0]
        assert list(m) == [NO_MOVE] * 3 and list(nodes) == [1, 1, 0]
        assert np.isnan(v[2])
    v0, m0 = xu.oracle_search(b[:2], w[:2], t[:2], weights, 3)
    assert np.array_equal(v[:2].astype(np.float64), v0) and list(m0) == [NO_MOVE] * 2


@pytest.mark.parametrize("depth", [1, 2, 3, 4])
def test_ties_take_the_lowest_square(oracle, depth):
    """with a table of weights in -2..2 root moves often tie: the move is the lowest square whose subtree reaches the
    value, although the root tries its moves best shallow score first from depth 3"""
    b, w, t = xu.spread(oracle, 1, 900 + depth, lo=8, hi=50)
    weights = xu.weights40(np.random.RandomState(depth).randint(-2, 3, size=(4, 10)))
    v, m, _ = xu.host_search(b, w, t, weights, depth)
    ties = 0
    for i in range(b.size):
        if m[i] >= 64:
            continue
        child = xu.oracle_children(b[i], w[i], t[i], weights, depth)
        best = np.nanmax(child)
        reach = np.nonzero(child == best)[0]
        assert v[i] == best and m[i] == reach.min()
        ties += reach.size > 1
    assert ties >= 5


@pytest.mark.parametrize("table", ["default", "int7"])
def test_depth_1_is_the_arg_max_of_the_children(oracle, spread, table):
    b, w, t = (a[::2] for a in spread)
    weights = TABLES[table]()
    v, m, nodes = xu.host_search(b, w, t, weights, 1)
    for i in range(b.size):
        squares, cb, cw = xu.successors(oracle, b[i], w[i], t[i])
        if not squares:
            continue
        s = oracle.evaluate(cb, cw, np.full(len(squares), t[i], np.uint8), weights)
        k = int(np.argmax(s))                                         # the first maximum: the lowest square
        assert (m[i], v[i]) == (squares[k], s[k]) and nodes[i] == 1 + len(squares)


def test_argument_validation_needs_no_gpu():
    from subproc_b200 import _lib
    L = _lib.lib()
    ws = L.othello_search_workspace_bytes()
    assert ws > 0
    buf = (ctypes.c_uint64 * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert L.othello_search(None, None, None, None, 1, None, None, None, 0, None, 0, None) == 0     # n = 0: no-op
    assert L.othello_search(p, p, None, p, 0, p, p, None, 4, p, ws, None) == -1                     # depth 0
    assert L.othello_search(p, p, None, p, 13, p, p, None, 4, p, ws, None) == -1                    # depth 13
    assert L.othello_search(p, p, None, p, 13, p, p, None, 0, p, ws, None) == -1                    # ... even for n = 0
    assert L.othello_search(p, p, None, p, 4, p, p, None, 4, p, ws - 1, None) == -2                 # workspace too small
    assert L.othello_search(p, p, None, None, 4, p, p, None, 4, p, ws, None) == -1                  # weights missing
    assert L.othello_search(p, p, None, p, 4, p, p, None, -1, p, ws, None) == -1                    # n < 0
