"""othello_search on the device (ops.search): bit-exact against the host build of csrc/midgame.cuh for float weights,
equal to the reference minimax of tests/search_oracle.c for integer weights, depth 1 equal to the greedy kernel,
results independent of the batch and the stream; the lock-step games of GameRunner with a search engine, and the
Edax-protocol engine's --policy search."""
import numpy as np
import pytest
import torch

import search_util as xu
import solve_util as su
from gpu_util import DEV, dev_bits, dev_u8
from search_util import BLACK, WHITE, PASS, NO_MOVE
from subproc_b200 import ops

pytestmark = pytest.mark.gpu


def dev_w(weights):
    return torch.from_numpy(xu.weights40(weights)).to(DEV)


def gpu_search(b, w, t, weights, depth):
    v, m, n = ops.search(dev_bits(b), dev_bits(w), dev_w(weights), depth, turn=dev_u8(t), nodes=True)
    return v.cpu().numpy(), m.cpu().numpy(), n.cpu().numpy()


@pytest.fixture(scope="module")
def wide(oracle):
    """~10^4 positions from 0..56 empties, with must-pass and game-over roots"""
    b, w, t = xu.spread(oracle, 170, 3000)
    (pb, pw, pt), (ob, ow, ot) = su.special_positions(oracle, 60, 3100)
    return tuple(np.concatenate(x) for x in zip((b, w, t), (pb, pw, pt), (ob, ow, ot)))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("depth", [1, 2, 3, 4, 5, 6])
def test_bit_exact_against_the_host_build_for_float_weights(wide, seed, depth):
    b, w, t = wide
    assert b.size > 9000 and np.any(t == WHITE)
    weights = xu.float_weights(seed)
    v, m, n = gpu_search(b, w, t, weights, depth)
    hv, hm, hn = xu.host_search(b, w, t, weights, depth)
    assert np.array_equal(v.view(np.uint32), hv.view(np.uint32))
    assert np.array_equal(m, hm) and np.array_equal(n, hn.astype(np.int64))
    assert np.any(m == PASS) and np.any(m == NO_MOVE)


def test_score_equals_ops_evaluate_for_float_weights(wide):
    b, w, t = wide
    weights = xu.float_weights(3)
    own, opp = np.where(t == BLACK, b, w), np.where(t == BLACK, w, b)
    ev = ops.evaluate(dev_bits(b), dev_bits(w), dev_u8(t), dev_w(weights)).cpu().numpy()
    assert np.array_equal(ev.view(np.uint32), xu.host_score(own, opp, weights).view(np.uint32))


@pytest.mark.parametrize("table", ["default", "int7"])
def test_against_the_reference_for_integer_weights(oracle, table):
    weights = xu.default_weights() if table == "default" else xu.int_weights(7)
    b, w, t = xu.spread(oracle, 5, 3200)
    for depth in (1, 2, 3):
        v0, m0 = xu.oracle_search(b, w, t, weights, depth, pruned=False)
        v, m, _ = gpu_search(b, w, t, weights, depth)
        assert np.array_equal(v.astype(np.float64), v0) and np.array_equal(m, m0), depth
    b, w, t = (a[::4] for a in (b, w, t))
    for depth in (4, 5):
        v0, m0 = xu.oracle_search(b, w, t, weights, depth, pruned=True)
        v, m, _ = gpu_search(b, w, t, weights, depth)
        assert np.array_equal(v.astype(np.float64), v0) and np.array_equal(m, m0), depth


@pytest.mark.parametrize("table", ["int", "float"])
def test_depth_1_is_the_greedy_kernel(table):
    """~10^5 start positions: the search's move is the ply-0 move of the greedy kernel, its value the evaluation of
    that successor from the mover's side"""
    weights = dev_w(xu.int_weights(21) if table == "int" else xu.float_weights(21))
    po = ops.playout(2048, seed=77, device=DEV)
    rows = torch.arange(0, 60, 1, device=DEV)
    live = rows[:, None] <= po.nplies[None, :].long()
    b0, w0 = po.black[:60][live].contiguous(), po.white[:60][live].contiguous()
    turn0 = torch.where(rows[:, None].expand(-1, 2048)[live] % 2 == 0, BLACK, WHITE).to(torch.uint8).contiguous()
    assert b0.numel() > 100000
    g = ops.playout(b0.numel(), device=DEV, black0=b0, white0=w0, turn0=turn0, policy=ops.POLICY_GREEDY, weights=weights,
                    t_max=1)
    v, m, _ = ops.search(b0, w0, weights, 1, turn=turn0)
    moved = g.nplies > 0                                           # (a game-over start plays no ply)
    assert torch.equal(m[moved], g.move[0][moved]) and bool((m[~moved] == NO_MOVE).all())
    ev = ops.evaluate(g.black[1].contiguous(), g.white[1].contiguous(), turn0, weights)
    assert torch.equal(v[moved].view(torch.int32), ev[moved].view(torch.int32))
    assert bool((m == PASS).any())


def test_the_batch_and_the_stream_do_not_matter(wide):
    b, w, t = (a[::10] for a in wide)
    weights = xu.float_weights(4)
    v0, m0, n0 = gpu_search(b, w, t, weights, 5)
    for i in (0, 7, b.size - 1):                                   # alone
        v, m, n = gpu_search(b[i:i + 1], w[i:i + 1], t[i:i + 1], weights, 5)
        assert (v.view(np.uint32)[0], m[0], n[0]) == (v0.view(np.uint32)[i], m0[i], n0[i])
    rng = np.random.RandomState(5)
    idx = rng.randint(0, b.size, 1 << 16)                          # inside a shuffled batch of 2^16
    v, m, n = gpu_search(b[idx], w[idx], t[idx], weights, 5)
    assert np.array_equal(v.view(np.uint32), v0.view(np.uint32)[idx]) and np.array_equal(m, m0[idx])
    assert np.array_equal(n, n0[idx])
    db, dw, dt, wt = dev_bits(b[idx]), dev_bits(w[idx]), dev_u8(t[idx]), dev_w(weights)
    streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]     # two streams at once, a workspace each
    torch.cuda.synchronize()
    outs = []
    for s in streams:
        with torch.cuda.stream(s):
            outs.append(ops.search(db, dw, wt, 5, turn=dt, nodes=True))
    torch.cuda.synchronize()
    for v, m, n in outs:
        assert np.array_equal(v.cpu().numpy().view(np.uint32), v0.view(np.uint32)[idx])
        assert np.array_equal(m.cpu().numpy(), m0[idx]) and np.array_equal(n.cpu().numpy(), n0[idx])


def test_arguments():
    e = torch.empty(0, dtype=torch.int64, device=DEV)
    v, m, n = ops.search(e, e, dev_w(xu.default_weights()), 3, nodes=True)
    assert v.numel() == 0 and m.numel() == 0 and n.numel() == 0
    for depth in (0, 13):
        with pytest.raises(ValueError):
            ops.search(e, e, dev_w(xu.default_weights()), depth)
    b, w = dev_bits([ops.START_BLACK, 3]), dev_bits([ops.START_WHITE, 6])
    v, m, _ = ops.search(b, w, dev_w(xu.default_weights()), 2)
    v2, m2, _ = ops.search(b, w, dev_w(xu.default_weights()), 2, turn=dev_u8([BLACK, BLACK]))
    assert int(m[0]) == int(m2[0]) and float(v[0]) == float(v2[0])
    assert torch.isnan(v[1]) and int(m[1]) == NO_MOVE


def referee_game(oracle, engines):
    """the moves of one game from the standard opening, each chosen by the reference search of the engine to move:
    engines = {colour: (weights, depth)}; returns [(black, white, turn, move)] and the final position"""
    b, w, turn = ops.START_BLACK, ops.START_WHITE, BLACK
    plies = []
    while not oracle.game_over([b], [w])[0]:
        weights, depth = engines[turn]
        _, m = xu.oracle_search([b], [w], [turn], weights, depth, pruned=depth > 3, threads=1)
        plies.append((b, w, turn, int(m[0])))
        nb, nw, nt, _, _, _ = oracle.step([b], [w], [turn], [len(plies) - 1], [int(m[0])])
        b, w, turn = int(nb[0]), int(nw[0]), int(nt[0])
    return plies, (b, w)


def test_lock_step_games_replay_against_the_reference(oracle):
    from subproc_b200.game_runner import GameRunner, Engine
    w1, w2 = xu.int_weights(31), xu.int_weights(32)
    ref, ref_final = referee_game(oracle, {BLACK: (w1, 3), WHITE: (w2, 1)})
    runner = GameRunner(Engine('search', w1, depth=3), Engine('greedy', w2), device=DEV)
    po = runner.play_games(3)
    n = len(ref)
    assert po.nplies.cpu().tolist() == [n] * 3
    assert ops.bits_numpy(po.final_black).tolist() == [ref_final[0]] * 3
    assert ops.bits_numpy(po.final_white).tolist() == [ref_final[1]] * 3
    assert po.move[:n, 0].cpu().tolist() == [m for _, _, _, m in ref]
    assert ops.bits_numpy(po.black[:n, 0]).tolist() == [b for b, _, _, _ in ref]
    assert ops.bits_numpy(po.white[:n, 0]).tolist() == [w for _, w, _, _ in ref]
    # White searches, Black is greedy, and the colours' tables swapped
    ref2, _ = referee_game(oracle, {BLACK: (w2, 1), WHITE: (w1, 2)})
    po2 = GameRunner(Engine('greedy', w2), Engine('search', w1, depth=2), device=DEV).play_games(1)
    assert po2.move[:len(ref2), 0].cpu().tolist() == [m for _, _, _, m in ref2]
    # learn_accumulate on the lock-step Playout = on a Playout rebuilt from the reference trajectory
    acc = ops.learn_accumulate(po)
    tb = np.array([b for b, _, _, _ in ref] + [ref_final[0]] * (po.t_max + 1 - n), np.uint64)
    tw = np.array([w for _, w, _, _ in ref] + [ref_final[1]] * (po.t_max + 1 - n), np.uint64)
    rebuilt = ops.Playout(3, po.t_max, dev_bits(np.repeat(tb, 3)).view(-1, 3).contiguous(),
                          dev_bits(np.repeat(tw, 3)).view(-1, 3).contiguous(), None,
                          torch.full((3,), n, dtype=torch.int32, device=DEV),
                          dev_bits([ref_final[0]] * 3), dev_bits([ref_final[1]] * 3))
    assert torch.equal(acc, ops.learn_accumulate(rebuilt))


def test_lock_step_games_from_start_positions_and_refusals(oracle):
    from subproc_b200.game_runner import GameRunner, Engine, play_search_games
    b, w, t = (a[:64] for a in xu.spread(oracle, 2, 3300, lo=20, hi=50))
    wt = dev_w(xu.int_weights(33))
    po = play_search_games(b.size, wt, 2, wt, 2, DEV, black0=dev_bits(b), white0=dev_bits(w), turn0=dev_u8(t))
    # every recorded move is the search's move in the recorded position
    nplies = po.nplies.cpu().numpy()
    for k in range(int(nplies.max())):
        g = np.nonzero(nplies > k)[0]
        turn_k = np.where((k % 2 == 0) == (t[g] == BLACK), BLACK, WHITE).astype(np.uint8)
        _, m, _ = ops.search(po.black[k][g].contiguous(), po.white[k][g].contiguous(), wt, 2, turn=dev_u8(turn_k))
        assert torch.equal(m, po.move[k][g])
    assert bool(oracle.game_over(ops.bits_numpy(po.final_black), ops.bits_numpy(po.final_white)).all())
    for bad in ((Engine('search', xu.int_weights(1), depth=2), Engine('random')),
                (Engine('search', xu.int_weights(1), depth=2), Engine('greedy', xu.int_weights(1), random_plies=4))):
        with pytest.raises(ValueError):
            GameRunner(*bad, device=DEV)
    with pytest.raises(ValueError):
        GameRunner(Engine('search', xu.int_weights(1), depth=2), Engine('greedy', xu.int_weights(1)), device=DEV,
                   n_rand_hands_for_black=2)
    from subproc_b200 import match
    assert match.engine_from_spec('search6').depth == 6


def test_engine_processes_search_then_solve():
    """two `edax_engine --policy search --depth 3 --exact 14` processes play a full game under the reference's
    Player protocol: every move with more than 14 empties is ops.search's, every later one ops.solve's"""
    import sys
    from test_gpu_next_rows import Player
    from subproc_b200 import board, parameter
    py = sys.executable
    cmd = "%s -m subproc_b200.edax_engine --policy search --depth 3 --exact 14 --name s%d"
    black, white = Player(cmd % (py, 1)), Player(cmd % (py, 2))
    black.init(); white.init()
    weights = dev_w(parameter.ProgressPositionMovesParameter().weights_table())
    ref = board.Board()
    searched = solved = 0
    while not ref.is_game_over():
        attacker, defender = (black, white) if ref.turn == board.Black else (white, black)
        own, opp = ref._pair(ref.turn)
        hand = attacker.go().lower()
        if 64 - bin(own | opp).count("1") > 14:
            _, m, _ = ops.search(dev_bits([own]), dev_bits([opp]), weights, 3)
            searched += 1
        else:
            _, m, _ = ops.solve(dev_bits([own]), dev_bits([opp]))
            solved += 1
        s = int(m[0])
        assert hand == ('ps' if s == PASS else ref.handstr_from_coord(s & 7, s >> 3).lower())
        assert ref.put_s(hand) >= 0
        assert defender.play(hand) == hand
    assert searched >= 40 and solved >= 10
    black.end_process(); white.end_process()
    assert black.proc.returncode == 0 and white.proc.returncode == 0
