"""Move values on the CPU: the host build of csrc/move_values.cuh (the function the kernels run per (position, move))
against the references of tests/search_oracle.c and tests/solve_oracle.c, row by row; the identities with the host
builds of othello_search and othello_solve (row maximum and lowest arg-max); and the argument checks of
othello_search_moves / othello_solve_moves through the built library (no device needed)."""
import ctypes

import numpy as np
import pytest

import move_values_util as mu
import search_util as xu
import solve_util as su
from search_util import BLACK, WHITE, PASS, NO_MOVE

REFUSED = mu.REFUSED


@pytest.fixture(scope="module")
def spread(oracle):
    return xu.spread(oracle, 5, 500)


@pytest.mark.parametrize("table", ["int7", "int8"])
@pytest.mark.parametrize("depth", [1, 2, 3, 4, 5])
def test_search_rows_equal_the_reference(oracle, spread, table, depth):
    b, w, t = spread if depth <= 3 else (a[::4] for a in spread)
    weights = xu.int_weights(int(table[3:]))
    ref, m0 = mu.oracle_rows(b, w, t, weights, depth)
    values, nodes = mu.host_search_moves(b, w, t, weights, depth)
    assert np.array_equal(values.astype(np.float64), ref, equal_nan=True), depth
    # the NaN pattern: the legal squares, and the pass column of the must-pass roots
    has = mu.legal_slots(mu.legal_masks(oracle, b, w, t))
    has[:, 64] = m0 == PASS
    assert np.array_equal(~np.isnan(values), has)
    assert np.all(nodes[has] >= 1) and np.all(nodes[~has] == 0)
    assert np.any(m0 == PASS) and np.any(m0 == NO_MOVE)


@pytest.mark.parametrize("depth", [1, 2, 3, 4, 5, 6])
def test_search_row_max_is_the_search(spread, depth):
    b, w, t = spread if depth <= 4 else (a[::2] for a in spread)
    for seed in (1, 2):
        weights = xu.float_weights(seed)
        v, m, _ = xu.host_search(b, w, t, weights, depth)
        values, _ = mu.host_search_moves(b, w, t, weights, depth)
        rv, rm = mu.row_max_search(values)
        over = m == NO_MOVE
        assert np.array_equal(rv[~over].view(np.uint32), v[~over].view(np.uint32)) and np.array_equal(rm, m)
        assert np.all(np.isnan(values[over])) and not np.any(np.signbit(values[values == 0]))


@pytest.mark.parametrize("table", ["default", "float"])
def test_search_depth_1_is_the_evaluation_of_each_successor(oracle, spread, table):
    b, w, t = (a[::2] for a in spread)
    weights = xu.default_weights() if table == "default" else xu.float_weights(5)
    values, nodes = mu.host_search_moves(b, w, t, weights, 1)
    for i in range(b.size):
        squares, cb, cw = xu.successors(oracle, b[i], w[i], t[i])
        own, opp = (cb, cw) if t[i] == BLACK else (cw, cb)
        if squares:
            assert np.array_equal(values[i, squares].view(np.uint32), xu.host_score(own, opp, weights).view(np.uint32))
            assert np.all(nodes[i, squares] == 1)


def test_search_rows_of_refused_and_finished_positions():
    """full boards (game over) and overlapping colours: every entry NaN with 0 nodes; the start: its four moves"""
    full = (1 << 64) - 1
    b = np.array([0x00000000FFFFFFFF, 0x00000000FFFFFFFF, 3, 0x0000000810000000], np.uint64)
    w = np.array([full & ~0x00000000FFFFFFFF, full & ~0x00000000FFFFFFFF, 6, 0x0000001008000000], np.uint64)
    t = np.array([BLACK, WHITE, BLACK, BLACK], np.uint8)
    for depth in (1, 6, 12):
        values, nodes = mu.host_search_moves(b, w, t, xu.int_weights(9), depth)
        assert np.all(np.isnan(values[:3])) and np.all(nodes[:3] == 0)
        assert np.flatnonzero(~np.isnan(values[3])).tolist() == [19, 26, 37, 44]


@pytest.fixture(scope="module")
def endgames(oracle):
    """0..12 empties, must-pass roots at 12 empties and up to 12 empties, game-over roots, and the constructed cases
    of solve_util (24 empties with a root pass and a three-way tie, 25 empties, the start, overlap, full boards)"""
    parts = [su.positions_with_empties(oracle, e, 6, 5000 + e) for e in range(0, 13)]
    parts.append(tuple(np.array(a, np.uint64) for a in zip(*su.MUST_PASS_12)) +
                 (np.full(len(su.MUST_PASS_12), BLACK, np.uint8),))
    parts += list(su.special_positions(oracle, 10, 5100, max_empties=12))
    cases = su.constructed_positions()
    parts.append(tuple(np.array([c[k] for c in cases], dt) for k, dt in ((0, np.uint64), (1, np.uint64), (2, np.uint8))))
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def test_solve_rows_equal_the_reference(oracle, endgames):
    b, w, t = endgames
    values, nodes = mu.host_solve_moves(b, w, t)
    v0, m0 = su.oracle_solve(b, w, t, pruned=True)
    checked = 0
    for i in range(b.size):
        row = values[i]
        refused = (int(b[i]) & int(w[i])) != 0 or su.empties([b[i]], [w[i]])[0] > 24
        squares, cb, cw = ([], None, None) if refused else xu.successors(oracle, b[i], w[i], t[i])
        expect = np.full(65, REFUSED, np.int32)
        if squares:
            cv, _ = su.oracle_solve(cb, cw, np.full(len(squares), WHITE if t[i] == BLACK else BLACK, np.uint8),
                                    pruned=True)
            expect[squares] = -cv
            checked += len(squares)
        elif m0[i] == PASS:
            expect[64] = v0[i]
        assert np.array_equal(row, expect), i
        assert np.array_equal(nodes[i] > 0, expect != REFUSED), i
    assert checked > 250 and np.any(m0 == PASS) and np.any((m0 == NO_MOVE) & (v0 != REFUSED))


def test_solve_row_max_is_the_solver(endgames):
    b, w, t = endgames
    values, _ = mu.host_solve_moves(b, w, t)
    v, m, _ = su.host_solve(b, w, t)
    rv, rm = mu.row_max_solve(values)
    none = m == NO_MOVE                                     # game over or refused: the whole row is REFUSED
    assert np.array_equal(rv[~none], v[~none]) and np.array_equal(rm, m)
    assert np.all(values[none] == REFUSED)


def test_argument_validation_needs_no_gpu():
    from subproc_b200 import _lib
    L = _lib.lib()
    sws, ews = L.othello_search_workspace_bytes(), L.othello_solve_workspace_bytes()
    buf = (ctypes.c_uint64 * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    search = L.othello_search_moves
    assert search(None, None, None, None, 1, None, None, 0, None, 0, None) == 0          # n = 0: no-op
    assert search(p, p, None, p, 0, p, None, 4, p, sws, None) == -1                     # depth 0
    assert search(p, p, None, p, 13, p, None, 4, p, sws, None) == -1                    # depth 13
    assert search(p, p, None, p, 13, p, None, 0, p, sws, None) == -1                    # ... even for n = 0
    assert search(p, p, None, p, 4, p, None, -1, p, sws, None) == -1                    # n < 0
    assert search(p, p, None, None, 4, p, None, 4, p, sws, None) == -1                  # weights missing
    assert search(None, p, None, p, 4, p, None, 4, p, sws, None) == -1                  # black missing
    assert search(p, p, None, p, 4, None, None, 4, p, sws, None) == -1                  # values missing
    assert search(p, p, None, p, 4, p, None, 4, None, sws, None) == -1                  # workspace missing
    assert search(p, p, None, p, 4, p, None, 4, p, sws - 1, None) == -2                 # workspace too small
    solve = L.othello_solve_moves
    assert solve(None, None, None, None, None, 0, None, 0, None) == 0                   # n = 0: no-op
    assert solve(p, p, None, p, None, -1, p, ews, None) == -1                           # n < 0
    assert solve(p, None, None, p, None, 4, p, ews, None) == -1                         # white missing
    assert solve(p, p, None, None, None, 4, p, ews, None) == -1                         # values missing
    assert solve(p, p, None, p, None, 4, None, ews, None) == -1                         # workspace missing
    assert solve(p, p, None, p, None, 4, p, ews - 1, None) == -2                        # workspace too small
