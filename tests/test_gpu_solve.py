"""othello_solve on the device (ops.solve) against the reference solvers of tests/solve_oracle.c: values and moves
equal, refused positions flagged, per-position node counts independent of the batch, and the Edax-protocol engine's
--exact mode playing perfect endgames."""
import functools
import io
import re

import numpy as np
import pytest
import torch

import solve_util as su
from gpu_util import DEV, dev_bits, dev_u8
from solve_util import BLACK, WHITE, PASS, NO_MOVE, REFUSED
from subproc_b200 import ops

pytestmark = pytest.mark.gpu


def gpu_solve(b, w, t, nodes=False):
    v, m, n = ops.solve(dev_bits(b), dev_bits(w), dev_u8(t), nodes=nodes)
    return v.cpu().numpy(), m.cpu().numpy(), (n.cpu().numpy() if nodes else None)


def cat(*parts):
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


@functools.lru_cache(maxsize=None)
def cheapest(oracle, e, k, seed):
    """the k of 40 sampled positions with e empties that the search solves with the fewest nodes, in sample order (the
    reference's unordered alpha-beta takes minutes on some 16-empty positions; the seeds below pick fast ones)"""
    b, w, t = su.positions_with_empties(oracle, e, 40, seed)
    _, _, nodes = su.host_solve(b, w, t)
    idx = np.sort(np.argsort(nodes, kind="stable")[:k])
    return b[idx], w[idx], t[idx]


def test_values_and_moves_against_minimax_0_to_10_empties(oracle):
    b, w, t = cat(*[su.positions_with_empties(oracle, e, 40, 1000 + e) for e in range(0, 11)])
    b2, w2, t2 = su.positions_before_pass(oracle, 10, 40, 1100)          # passes inside the tree
    b, w, t = np.concatenate([b, b2]), np.concatenate([w, w2]), np.concatenate([t, t2])
    v0, m0 = su.oracle_solve(b, w, t, pruned=False)
    v, m, _ = gpu_solve(b, w, t)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)


SEEDED_K = ((13, 6), (14, 4), (15, 3), (16, 2))      # empties, positions checked against orc_solve_ab


def test_values_and_moves_against_alphabeta_12_to_16_empties(oracle):
    mp12 = tuple(np.array(a, np.uint64) for a in zip(*su.MUST_PASS_12)) + (np.full(len(su.MUST_PASS_12), BLACK, np.uint8),)
    b, w, t = cat(su.positions_with_empties(oracle, 12, 48, 1212), mp12,
                  *[cheapest(oracle, e, k, 1200 + e) for e, k in SEEDED_K])
    v0, m0 = su.oracle_solve(b, w, t, pruned=True)
    v, m, _ = gpu_solve(b, w, t)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)


def test_constructed_positions():
    cases = su.constructed_positions()
    b, w, t = (np.array([c[k] for c in cases], dtype) for k, dtype in ((0, np.uint64), (1, np.uint64), (2, np.uint8)))
    v0, m0 = su.oracle_solve(b, w, t, pruned=False)
    v, m, nodes = gpu_solve(b, w, t, nodes=True)
    assert np.array_equal(v, v0) and np.array_equal(m, m0)
    hv, hm, hn = su.host_solve(b, w, t)
    assert np.array_equal(nodes, hn.astype(np.int64))                    # the same search as the host build


@pytest.fixture(scope="module")
def mixed(oracle):
    """one batch: 0..16 empties (with reference values), 17 and 18 empties (value -999: no reference), 24 empties with
    a root pass and a three-way tie (reference values), refused positions (25 empties and more, overlapping colours),
    must-pass and game-over roots; and its solution in one call (value, move, nodes).  Positions from random games with
    19..24 empties take minutes in one lane, so the deep end of the range is the constructed 24-empty pair."""
    parts = [su.positions_with_empties(oracle, e, 8, 2000 + e) for e in range(0, 13)]
    parts += [tuple(a[:2] for a in cheapest(oracle, e, k, 1200 + e)) for e, k in SEEDED_K]
    parts += [tuple(np.array(a, dtype) for a, dtype in zip(zip(*[c[:3] for c in su.constructed_positions()
                                                                 if c[3].startswith("24 empties")]),
                                                             (np.uint64, np.uint64, np.uint8)))]
    (pb, pw, pt), (ob, ow, ot) = su.special_positions(oracle, 12, 2100, max_empties=16)
    assert pb.size >= 6 and ob.size == 12
    b, w, t = cat(*parts, (pb, pw, pt), (ob, ow, ot))
    v_ref, m_ref = su.oracle_solve(b, w, t, pruned=True)
    deep = cat(su.positions_with_empties(oracle, 17, 3, 2217),      # + an 18-empty position of a random game that solves fast
               (np.array([0x8b573f1f5b7d7e7e], np.uint64), np.array([0x0000000004020100], np.uint64), np.array([BLACK], np.uint8)))
    start = (np.array([0x0000000810000000], np.uint64), np.array([0x0000001008000000], np.uint64), np.array([BLACK], np.uint8))
    over25 = su.positions_with_empties(oracle, 25, 4, 2300)
    overlap = (np.array([3, 0xFF], np.uint64), np.array([6, 0x1FF80], np.uint64), np.array([BLACK, WHITE], np.uint8))
    refused = cat(start, over25, overlap)
    b, w, t = cat((b, w, t), deep, refused)
    v_ref = np.concatenate([v_ref, np.full(deep[0].size, -999), np.full(refused[0].size, REFUSED)]).astype(np.int32)
    m_ref = np.concatenate([m_ref, np.zeros(deep[0].size), np.full(refused[0].size, NO_MOVE)]).astype(np.uint8)
    return (b, w, t, v_ref, m_ref), gpu_solve(b, w, t, nodes=True)


def test_mixed_batch(mixed):
    (b, w, t, v_ref, m_ref), (v, m, nodes) = mixed
    known = v_ref != -999
    assert np.array_equal(v[known], v_ref[known]) and np.array_equal(m[known], m_ref[known])
    deep = ~known
    assert np.all(np.abs(v[deep]) <= 64) and np.all(m[deep] <= PASS)
    refused = v_ref == REFUSED
    assert np.all(nodes[refused] == 0) and np.all(nodes[~refused] >= 1)
    assert np.any(m == PASS) and np.any((m == NO_MOVE) & ~refused)


@pytest.mark.parametrize("size", [1, 31, 33, 4000])
def test_batch_sizes_permutations_and_splits(mixed, size):
    """the positions of the mixed batch in another order, in calls of `size` positions: identical values, moves and
    per-position node counts; without the nodes output the values and moves do not change.  The small sizes take
    four calls; 4000 tiles the batch, so every position is solved again in another place."""
    (b, w, t, _, _), (v0, m0, n0) = mixed
    rng = np.random.RandomState(size)
    if size >= b.size:
        idx = rng.permutation(np.tile(np.arange(b.size), -(-size // b.size)))[:size]
        idx[:b.size] = rng.permutation(b.size)
    else:
        idx = rng.permutation(b.size)[:4 * size]
    vs, ms, ns = [], [], []
    for lo in range(0, idx.size, size):
        part = idx[lo:lo + size]
        v, m, n = gpu_solve(b[part], w[part], t[part], nodes=True)
        vs.append(v); ms.append(m); ns.append(n)
    v, m, n = np.concatenate(vs), np.concatenate(ms), np.concatenate(ns)
    assert np.array_equal(v, v0[idx]) and np.array_equal(m, m0[idx]) and np.array_equal(n, n0[idx])
    part = idx[:size]
    v1, m1, _ = gpu_solve(b[part], w[part], t[part], nodes=False)
    assert np.array_equal(v1, v0[part]) and np.array_equal(m1, m0[part])


def test_turn_none_means_black_and_empty_batch():
    b, w = dev_bits([0x00000000FFFFFFFF]), dev_bits([0xFFFFFFFF00000000 & ~(1 << 63)])
    v, m, _ = ops.solve(b, w)
    v2, m2, _ = ops.solve(b, w, dev_u8([BLACK]))
    assert int(v[0]) == int(v2[0]) and int(m[0]) == int(m2[0])
    e = torch.empty(0, dtype=torch.int64, device=DEV)
    v, m, n = ops.solve(e, e, nodes=True)
    assert v.numel() == 0 and m.numel() == 0 and n.numel() == 0


def _engine_game(be_black, be_white):
    """a game between two in-process engines through the protocol: [(black, white, turn, hand played)]"""
    from subproc_b200.edax_engine import EdaxFrontEnd
    outs = {BLACK: io.StringIO(), WHITE: io.StringIO()}
    fes = {BLACK: EdaxFrontEnd(be_black, out=outs[BLACK]), WHITE: EdaxFrontEnd(be_white, out=outs[WHITE])}
    for fe in fes.values():
        fe.handle("init")
    played = []
    turn = BLACK
    while not be_black.b.is_game_over():
        b, w = be_black.b._black, be_black.b._white
        fes[turn].handle("go")
        hand = re.findall(r"plays ([A-Z][0-9]|PS)", outs[turn].getvalue())[-1]
        fes[WHITE if turn == BLACK else BLACK].handle(hand.lower())
        played.append((b, w, turn, hand))
        turn = WHITE if turn == BLACK else BLACK
        assert (be_black.b._black, be_black.b._white) == (be_white.b._black, be_white.b._white)
    return played


def _square(hand):
    return PASS if hand == 'PS' else (ord(hand[0].lower()) - ord('a')) + 8 * (int(hand[1]) - 1)


def test_engine_exact_mode_plays_perfect_endgames(oracle):
    """--exact 14 against the greedy engine, on either side: every move it played with at most 14 empties reaches
    the reference's perfect-play value of the position it was played in"""
    from subproc_b200 import parameter
    from subproc_b200.edax_engine import Backend
    weights = parameter.ProgressPositionMovesParameter().weights_table()
    roots, children = [], []
    for exact_side in (BLACK, WHITE):
        exact, greedy = Backend('greedy', weights, exact_empties=14), Backend('greedy', weights)
        players = (exact, greedy) if exact_side == BLACK else (greedy, exact)
        for b, w, turn, hand in _engine_game(*players):
            if turn != exact_side or 64 - bin(b | w).count("1") > 14 or hand == 'PS':
                continue
            cb, cw, _, ret = oracle.put([b], [w], turn, [_square(hand)])
            assert ret[0] > 0
            roots.append((b, w, turn))
            children.append((int(cb[0]), int(cw[0]), WHITE if turn == BLACK else BLACK))
    assert len(roots) >= 10
    v_root, _ = su.oracle_solve(*zip(*roots), pruned=True)
    v_child, _ = su.oracle_solve(*zip(*children), pruned=True)
    assert np.array_equal(-v_child, v_root)


def test_engine_without_exact_plays_as_before(oracle):
    """no --exact: the greedy engine's game is the oracle's greedy game, move for move"""
    from subproc_b200 import parameter
    from subproc_b200.edax_engine import Backend
    weights = parameter.ProgressPositionMovesParameter().weights_table()
    played = _engine_game(Backend('greedy', weights), Backend('greedy', weights))
    ref = oracle.playout(0, 0, 1, policy=1, weights=weights.astype(np.float64))
    assert len(played) == int(ref['nplies'][0])
    assert [_square(h) for _, _, _, h in played] == [int(x) for x in ref['move'][:len(played), 0]]
