"""othello_search_moves / othello_solve_moves on the device (ops.search_moves, ops.solve_moves): rows bit-exact
against the host build of csrc/move_values.cuh, equal to the references, depth 1 = the evaluation of every successor,
row maximum and lowest arg-max = ops.search / ops.solve, minus ops.solve of every child, sentinels, and results
independent of the batch, the order, the split into calls and the stream."""
import numpy as np
import pytest
import torch

import move_values_util as mu
import search_util as xu
import solve_util as su
from gpu_util import DEV, dev_bits, dev_u8
from search_util import BLACK, WHITE, PASS, NO_MOVE
from subproc_b200 import ops

pytestmark = pytest.mark.gpu

REFUSED = ops.SOLVE_REFUSED


def dev_w(weights):
    return torch.from_numpy(xu.weights40(weights)).to(DEV)


def gpu_search_moves(b, w, t, weights, depth):
    v, n = ops.search_moves(dev_bits(b), dev_bits(w), dev_w(weights), depth, turn=dev_u8(t), nodes=True)
    return v.cpu().numpy(), n.cpu().numpy()


def gpu_solve_moves(b, w, t):
    v, n = ops.solve_moves(dev_bits(b), dev_bits(w), turn=dev_u8(t), nodes=True)
    return v.cpu().numpy(), n.cpu().numpy()


def children(b, w, t):
    """every (position, legal square) pair of device positions, on the device: (index, square, child black, child
    white, child's mover)"""
    own, opp = torch.where(t == BLACK, b, w), torch.where(t == BLACK, w, b)
    legal = ops.legal(own, opp)
    bit = torch.arange(64, device=b.device)
    pairs = torch.nonzero(((legal[:, None] >> bit[None, :]) & 1) != 0)
    i, s = pairs[:, 0].contiguous(), pairs[:, 1].contiguous()
    f = ops.flips(own[i].contiguous(), opp[i].contiguous(), s.to(torch.uint8))
    c_own = own[i] | f | torch.bitwise_left_shift(torch.ones_like(f), s)
    c_opp = opp[i] & ~f
    black_moved = t[i] == BLACK
    cb, cw = torch.where(black_moved, c_own, c_opp), torch.where(black_moved, c_opp, c_own)
    return i, s, cb.contiguous(), cw.contiguous(), torch.where(black_moved, WHITE, BLACK).to(torch.uint8)


def row_max(values, sentinel_is_nan):
    """(max, lowest arg-max, has a value) of each device row"""
    has_entry = ~torch.isnan(values) if sentinel_is_nan else values != REFUSED
    low = -torch.inf if sentinel_is_nan else -1000
    v = torch.where(has_entry, values, torch.full_like(values, low))
    arg = torch.argmax(v, dim=1)                                   # the first maximum: the lowest index reaching it
    return v.gather(1, arg[:, None])[:, 0], arg, has_entry.any(dim=1)


@pytest.fixture(scope="module")
def wide(oracle):
    """~10^4 positions from 0..56 empties, with must-pass and game-over roots"""
    b, w, t = xu.spread(oracle, 170, 6000)
    (pb, pw, pt), (ob, ow, ot) = su.special_positions(oracle, 60, 6100)
    return tuple(np.concatenate(x) for x in zip((b, w, t), (pb, pw, pt), (ob, ow, ot)))


@pytest.mark.parametrize("depth", [1, 2, 3, 4, 5, 6])
def test_search_bit_exact_against_the_host_build_for_float_weights(wide, depth):
    b, w, t = wide
    assert b.size > 9000 and np.any(t == WHITE)
    weights = xu.float_weights(depth)
    v, n = gpu_search_moves(b, w, t, weights, depth)
    hv, hn = mu.host_search_moves(b, w, t, weights, depth)
    assert np.array_equal(v.view(np.uint32), hv.view(np.uint32)) and np.array_equal(n, hn.astype(np.int64))
    assert np.any(~np.isnan(v[:, 64])) and np.any(np.isnan(v).all(axis=1))


@pytest.mark.parametrize("table", ["default", "int7"])
def test_search_against_the_reference_for_integer_weights(oracle, table):
    weights = xu.default_weights() if table == "default" else xu.int_weights(7)
    b, w, t = xu.spread(oracle, 4, 6200)
    for depth in (1, 2, 3, 4):
        bb, ww, tt = (b, w, t) if depth <= 3 else (a[::3] for a in (b, w, t))
        ref, m0 = mu.oracle_rows(bb, ww, tt, weights, depth)
        v, _ = gpu_search_moves(bb, ww, tt, weights, depth)
        assert np.array_equal(v.astype(np.float64), ref, equal_nan=True), depth
        assert np.any(m0 == PASS) and np.any(m0 == NO_MOVE)


def test_search_depth_1_is_the_evaluation_of_every_successor(wide):
    b, w, t = dev_bits(wide[0]), dev_bits(wide[1]), dev_u8(wide[2])
    weights = dev_w(xu.float_weights(11))
    values, nodes = ops.search_moves(b, w, weights, 1, turn=t, nodes=True)
    i, s, cb, cw, _ = children(b, w, t)
    assert i.numel() > 50000
    ev = ops.evaluate(cb, cw, t[i].contiguous(), weights)           # side = the mover at the root
    assert torch.equal(values[i, s].view(torch.int32), ev.view(torch.int32))
    assert bool((nodes[i, s] == 1).all())


@pytest.fixture(scope="module")
def game_positions():
    """> 10^5 positions of 2048 seeded random games, every ply, both colours to move, must-pass and game-over ones"""
    po = ops.playout(2048, seed=91, device=DEV)
    rows = torch.arange(0, 61, 1, device=DEV)
    live = rows[:, None] <= po.nplies[None, :].long()
    b, w = po.black[:61][live].contiguous(), po.white[:61][live].contiguous()
    turn = torch.where(rows[:, None].expand(-1, 2048)[live] % 2 == 0, BLACK, WHITE).to(torch.uint8).contiguous()
    assert b.numel() > 100000
    return b, w, turn


@pytest.mark.parametrize("depth", [1, 2, 3, 4])
def test_search_row_max_is_ops_search(game_positions, depth):
    b, w, t = game_positions
    weights = dev_w(xu.float_weights(20 + depth))
    values, _ = ops.search_moves(b, w, weights, depth, turn=t)
    v, m, _ = ops.search(b, w, weights, depth, turn=t)
    best, arg, has = row_max(values, True)
    assert torch.equal(has, m != NO_MOVE) and bool((m == PASS).any()) and bool((m == NO_MOVE).any())
    assert torch.equal(best[has].view(torch.int32), v[has].view(torch.int32))
    assert torch.equal(arg[has].to(torch.uint8), m[has])
    assert bool(torch.isnan(values[~has]).all())


def cheap_endgames(oracle, e, k, seed):
    """k of 40 sampled positions with e empties: those with the fewest moves on both sides (a proxy for a small
    solve), in sample order"""
    b, w, t = su.positions_with_empties(oracle, e, 40, seed)
    own, opp = np.where(t == BLACK, b, w), np.where(t == BLACK, w, b)
    mob = lambda m: np.array([bin(int(x)).count("1") for x in m])
    cost = (mob(oracle.puttables(own, opp, BLACK)) + 1) * (mob(oracle.puttables(opp, own, BLACK)) + 1)
    idx = np.sort(np.argsort(cost, kind="stable")[:k])
    return b[idx], w[idx], t[idx]


# 20 empties (ranks 6-8 but a6, b6, g6, h6), White's one disc e5 among Black's ranks 1-5: Black's d6, e6 and f6 each take
# it and end the game, White to move must pass.  Positions of random games with 19 or more empties cost millions of
# nodes in one lane (minutes on the device), so the deep end of the range is this pair, 17 empties from random games
# and the 18-empty position of test_gpu_solve.py that solves fast.
DEEP_20 = (((1 << 40) - 1) & ~su.bits('e5')) | su.bits('a6', 'b6', 'g6', 'h6'), su.bits('e5')


@pytest.fixture(scope="module")
def endgames(oracle):
    """12..20 empties (the larger, the fewer), must-pass and game-over roots, the constructed 24-empty pair"""
    parts = [su.positions_with_empties(oracle, 12, 64, 6312)]
    parts += [cheap_endgames(oracle, e, k, 6300 + e) for e, k in ((13, 16), (14, 16), (15, 8), (16, 8))]
    parts.append(su.positions_with_empties(oracle, 17, 3, 2217))
    parts.append((np.array([0x8b573f1f5b7d7e7e, DEEP_20[0], DEEP_20[0]], np.uint64),
                  np.array([0x0000000004020100, DEEP_20[1], DEEP_20[1]], np.uint64), np.array([BLACK, BLACK, WHITE], np.uint8)))
    parts.append(tuple(np.array(a, np.uint64) for a in zip(*su.MUST_PASS_12)) +
                 (np.full(len(su.MUST_PASS_12), BLACK, np.uint8),))
    parts += list(su.special_positions(oracle, 12, 6400, max_empties=16))
    parts.append(tuple(np.array(a, dt) for a, dt in zip(zip(*[c[:3] for c in su.constructed_positions()
                                                             if c[3].startswith("24 empties")]),
                                                         (np.uint64, np.uint64, np.uint8))))
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def test_solve_rows_are_minus_the_children_and_their_max_is_ops_solve(endgames):
    b, w, t = (dev_bits(endgames[0]), dev_bits(endgames[1]), dev_u8(endgames[2]))
    values, nodes = ops.solve_moves(b, w, turn=t, nodes=True)
    i, s, cb, cw, ct = children(b, w, t)
    cv, _, _ = ops.solve(cb, cw, ct)
    expect = torch.full_like(values, REFUSED)
    expect[i, s] = -cv
    v, m, _ = ops.solve(b, w, t)
    expect[:, 64] = torch.where(m == PASS, v, torch.full_like(v, REFUSED))
    assert torch.equal(values, expect)
    assert torch.equal(nodes > 0, expect != REFUSED)
    best, arg, has = row_max(values, False)
    assert torch.equal(has, m != NO_MOVE) and bool((m == PASS).any()) and bool((m == NO_MOVE).any())
    assert torch.equal(best[has], v[has]) and torch.equal(arg[has].to(torch.uint8), m[has])
    assert {12, 16, 20, 24} <= set(su.empties(endgames[0], endgames[1]).tolist())


def test_solve_rows_equal_the_host_build(endgames):
    keep = su.empties(endgames[0], endgames[1]) <= 16                # (the host build solves on the CPU)
    b, w, t = (a[keep] for a in endgames)
    v, n = gpu_solve_moves(b, w, t)
    hv, hn = mu.host_solve_moves(b, w, t)
    assert np.array_equal(v, hv) and np.array_equal(n, hn.astype(np.int64))


def test_sentinels_24_and_25_empties_and_overlap():
    cases = {c[3]: c[:3] for c in su.constructed_positions()}
    names = ["24 empties, root must pass", "24 empties, three moves tie", "too many empties: 25", "too many empties",
             "overlap", "full board", "game over, empties left"]
    b, w, t = (np.array([cases[k][j] for k in names], dt) for j, dt in ((0, np.uint64), (1, np.uint64), (2, np.uint8)))
    v, n = gpu_solve_moves(b, w, t)
    v0, m0 = su.oracle_solve(b[:2], w[:2], t[:2])
    assert np.flatnonzero(v[0] != REFUSED).tolist() == [64] and v[0, 64] == v0[0] and m0[0] == PASS
    assert np.flatnonzero(v[1] != REFUSED).tolist() == [43, 44, 45] and v[1].max() == v0[1]
    assert np.all(v[2:] == REFUSED) and np.all(n[2:] == 0)
    sv, sn = gpu_search_moves(b, w, t, xu.int_weights(3), 3)
    assert np.all(np.isnan(sv[4:])) and np.all(sn[4:] == 0)              # overlap, game over: all NaN
    assert np.flatnonzero(~np.isnan(sv[0])).tolist() == [64]


def test_turn_none_is_black_and_empty_batches():
    b, w = dev_bits([ops.START_BLACK, 0x00000000FFFFFFFF]), dev_bits([ops.START_WHITE, 0xFFFFFFFF00000000 & ~(1 << 63)])
    weights = dev_w(xu.default_weights())
    v1, _ = ops.search_moves(b, w, weights, 3)
    v2, _ = ops.search_moves(b, w, weights, 3, turn=dev_u8([BLACK, BLACK]))
    assert torch.equal(v1.nan_to_num(7.5).view(torch.int32), v2.nan_to_num(7.5).view(torch.int32))
    s1, _ = ops.solve_moves(b[1:], w[1:])
    s2, _ = ops.solve_moves(b[1:], w[1:], turn=dev_u8([BLACK]))
    assert torch.equal(s1, s2) and bool((s1 != REFUSED).any())
    e = torch.empty(0, dtype=torch.int64, device=DEV)
    v, n = ops.search_moves(e, e, weights, 2, nodes=True)
    assert v.shape == (0, 65) and n.shape == (0, 65)
    v, n = ops.solve_moves(e, e, nodes=True)
    assert v.shape == (0, 65) and n.shape == (0, 65)
    for depth in (0, 13):
        with pytest.raises(ValueError):
            ops.search_moves(e, e, weights, depth)


@pytest.mark.parametrize("kind", ["search", "solve"])
def test_batch_order_splits_and_streams_do_not_matter(wide, endgames, kind):
    """the same rows and node counts alone, in calls of 1, 31 and 33 positions of a shuffled order, in a shuffled
    batch of 2^16, with and without nodes, and on two streams at once"""
    weights = xu.float_weights(8)
    if kind == "search":
        b, w, t = (a[::10] for a in wide)
        run = lambda b, w, t, nodes=True: ops.search_moves(b, w, dev_w(weights), 5, turn=t, nodes=nodes)
    else:
        keep = su.empties(endgames[0], endgames[1]) <= 16
        b, w, t = (a[keep] for a in endgames)
        run = lambda b, w, t, nodes=True: ops.solve_moves(b, w, turn=t, nodes=nodes)
    bits = lambda v: v.view(torch.int32).cpu().numpy()
    v0, n0 = run(dev_bits(b), dev_bits(w), dev_u8(t))
    v0, n0 = bits(v0), n0.cpu().numpy()
    rng = np.random.RandomState(3)
    for size in (1, 31, 33):
        idx = rng.permutation(b.size)[:3 * size]
        for lo in range(0, idx.size, size):
            part = idx[lo:lo + size]
            v, n = run(dev_bits(b[part]), dev_bits(w[part]), dev_u8(t[part]))
            assert np.array_equal(bits(v), v0[part]) and np.array_equal(n.cpu().numpy(), n0[part])
    idx = rng.randint(0, b.size, 1 << 16)
    db, dw, dt = dev_bits(b[idx]), dev_bits(w[idx]), dev_u8(t[idx])
    v, n = run(db, dw, dt)
    assert np.array_equal(bits(v), v0[idx]) and np.array_equal(n.cpu().numpy(), n0[idx])
    v, n = run(db, dw, dt, nodes=False)
    assert n is None and np.array_equal(bits(v), v0[idx])
    streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]     # two streams at once, a workspace each
    torch.cuda.synchronize()
    outs = []
    for s in streams:
        with torch.cuda.stream(s):
            outs.append(run(db, dw, dt))
    torch.cuda.synchronize()
    for v, n in outs:
        assert np.array_equal(bits(v), v0[idx]) and np.array_equal(n.cpu().numpy(), n0[idx])
