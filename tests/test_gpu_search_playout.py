"""Search self-play on the device (othello_playout with OTHELLO_POLICY_SEARCH): depth 1 is the greedy kernel game for
game; without random plies the games are the lock-step games of play_search_games; with random plies, substitution and
a random opponent they replay against the host referee (tests/search_playout_util.py); results do not depend on the
batch, the launches or the stream; the learner's depth option; argument checks."""
import ctypes

import numpy as np
import pytest
import torch

import search_playout_util as pu
import search_util as xu
from gpu_util import DEV, dev_bits, dev_u8
from subproc_b200 import _lib, ops

pytestmark = pytest.mark.gpu

S, G, R = ops.POLICY_SEARCH, ops.POLICY_GREEDY, ops.POLICY_RANDOM


def dev_w(weights):
    return torch.from_numpy(xu.weights40(weights)).to(DEV)


def run(n, trajectory=True, **kw):
    """one playout with totals and summary: (Playout, totals int64 [4], summary int16 [n])"""
    totals = torch.zeros(4, dtype=torch.int64, device=DEV)
    summary = torch.empty(n, dtype=torch.int16, device=DEV)
    po = ops.playout(n, device=DEV, trajectory=trajectory, totals=totals, summary=summary, **kw)
    return po, totals, summary


def assert_same_games(a, b, t_max):
    """two Playouts: recorded rows t <= min(nplies, t_max), moves t < min(nplies, t_max), nplies, final positions"""
    assert torch.equal(a.nplies, b.nplies)
    assert torch.equal(a.final_black, b.final_black) and torch.equal(a.final_white, b.final_white)
    if a.black is None:
        return
    t = torch.arange(t_max + 1, device=DEV)[:, None]
    rows = t <= torch.clamp(a.nplies.long(), max=t_max)[None, :]
    assert torch.equal(a.black[rows], b.black[rows]) and torch.equal(a.white[rows], b.white[rows])
    if t_max > 0:
        moves = t[:-1] < torch.clamp(a.nplies.long(), max=t_max)[None, :]
        assert torch.equal(a.move[moves], b.move[moves])


def starts(n, seed):
    """n start positions from random playouts (rows 0..30), half of them with White to move"""
    po = ops.playout(n, seed=seed, device=DEV)
    t = torch.randint(0, 31, (n,), generator=torch.Generator().manual_seed(seed)).to(DEV)
    t = torch.minimum(t, po.nplies.long())
    g = torch.arange(n, device=DEV)
    turn = torch.where(g % 2 == 0, ops.BLACK, ops.WHITE).to(torch.uint8)
    return po.black[t, g].contiguous(), po.white[t, g].contiguous(), turn


CONFIGS = {
    "plain": dict(),
    "random_plies": dict(random_plies=6),
    "substitution": dict(random_plies=2, n_rand_black=3, n_rand_white=5),
    "random_white": dict(random_plies=1, policy_white=R),
    "random_black": dict(policy=R, policy_white="x", n_rand_white=3),
    "float_tables": dict(random_plies=4, tables="float"),
    "white_to_move": dict(start=True, n_rand_black=5),
    "t_max_0": dict(random_plies=6, t_max=0),
    "t_max_10": dict(random_plies=6, t_max=10),
    "no_trajectory": dict(random_plies=6, trajectory=False),
}


@pytest.mark.parametrize("n", [1, 4099, (1 << 16) + 3])
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_depth_1_is_the_greedy_kernel(name, n):
    c = dict(CONFIGS[name])
    tables = c.pop("tables", "int")
    w1, w2 = (xu.int_weights(61), xu.int_weights(62)) if tables == "int" else (xu.float_weights(61), xu.float_weights(62))
    kw = dict(seed=97, gid0=5000, weights=dev_w(w1), weights_white=dev_w(w2), t_max=c.pop("t_max", 120),
              trajectory=c.pop("trajectory", True))
    if c.pop("start", False):
        kw["black0"], kw["white0"], kw["turn0"] = starts(n, 98)
    kw.update(c)
    policy, policy_white = kw.pop("policy", "x"), kw.pop("policy_white", None)
    as_engine = lambda p, engine: engine if p == "x" else p       # "x": the side under test
    po_s, tot_s, sum_s = run(n, policy=as_engine(policy, S), policy_white=None if policy_white is None else
                             as_engine(policy_white, S), depth=1, **kw)
    po_g, tot_g, sum_g = run(n, policy=as_engine(policy, G), policy_white=None if policy_white is None else
                             as_engine(policy_white, G), **kw)
    assert_same_games(po_s, po_g, kw["t_max"])
    assert torch.equal(tot_s, tot_g) and torch.equal(sum_s, sum_g)
    assert int(tot_s[0]) == int(po_g.nplies.sum())


def openings(n, seed):
    """n 8-ply openings (Black to move: no game passes or ends in its first 8 plies)"""
    po = ops.playout(n, seed=seed, device=DEV)
    assert bool((po.nplies > 8).all())
    return po.black[8].contiguous(), po.white[8].contiguous()


@pytest.mark.parametrize("pairing", ["2-2", "4-greedy", "3-2_two_tables"])
def test_equal_to_lock_step_without_randomness(pairing):
    from subproc_b200.game_runner import play_search_games
    n = 512
    b0, w0 = openings(n, 71)
    wa, wb = dev_w(xu.int_weights(72)), dev_w(xu.float_weights(73))
    (pb, db, wtb), (pw, dw, wtw) = {
        "2-2": ((S, 2, wa), (S, 2, wa)),
        "4-greedy": ((S, 4, wa), (G, 1, wa)),
        "3-2_two_tables": ((S, 3, wa), (S, 2, wb)),
    }[pairing]
    po = ops.playout(n, seed=3, device=DEV, black0=b0, white0=w0, policy=pb, policy_white=pw, depth=db,
                     depth_white=dw if pw == S else None, weights=wtb, weights_white=wtw)
    ref = play_search_games(n, wtb, db, wtw, dw, DEV, black0=b0, white0=w0)
    assert_same_games(po, ref, po.t_max)


@pytest.mark.parametrize("config", ["2-3_subst", "3_vs_random", "random_vs_2"])
def test_full_replay_against_the_referee(oracle, config):
    n = 160
    w1, w2 = xu.int_weights(81), xu.int_weights(82)
    c = {
        "2-3_subst": dict(policy=S, policy_white=S, depth=2, depth_white=3, random_plies=4, n_rand_black=2,
                          n_rand_white=3),
        "3_vs_random": dict(policy=S, policy_white=R, depth=3, random_plies=2, n_rand_black=4),
        "random_vs_2": dict(policy=R, policy_white=S, depth=2, random_plies=0, n_rand_white=2),
    }[config]
    ref = pu.referee(oracle, n, seed=11, gid0=300, weights=w1, weights_white=w2, **c)
    po, tot, _ = run(n, seed=11, gid0=300, weights=dev_w(w1), weights_white=dev_w(w2), **c)
    check_against(po, tot, ref)


def check_against(po, tot, ref):
    nplies = po.nplies.cpu().numpy()
    assert np.array_equal(nplies, ref["nplies"])
    assert np.array_equal(ops.bits_numpy(po.final_black), ref["final_black"])
    assert np.array_equal(ops.bits_numpy(po.final_white), ref["final_white"])
    t = np.arange(po.t_max + 1)[:, None]
    rows = t <= nplies[None, :]
    assert np.array_equal(ops.bits_numpy(po.black)[rows], ref["black"][rows])
    assert np.array_equal(ops.bits_numpy(po.white)[rows], ref["white"][rows])
    moves = t[:-1] < nplies[None, :]
    assert np.array_equal(po.move.cpu().numpy()[moves], ref["move"][moves])
    assert tot.cpu().tolist() == ref["totals"].tolist()


def test_float_tables_replay_against_the_host_build(oracle):
    """every searched ply is the move of the host build of midgame.cuh, bit for bit"""
    n = 96
    w1, w2 = xu.float_weights(91), xu.float_weights(92)
    c = dict(policy=S, policy_white=S, depth=3, depth_white=2, random_plies=6, n_rand_black=3, n_rand_white=1)
    ref = pu.referee(oracle, n, seed=12, gid0=7, weights=w1, weights_white=w2, searcher=pu.host_searcher, **c)
    po, tot, _ = run(n, seed=12, gid0=7, weights=dev_w(w1), weights_white=dev_w(w2), **c)
    check_against(po, tot, ref)


def test_independent_of_batch_launches_and_streams():
    n = 1 << 16
    kw = dict(seed=21, policy=S, depth=2, random_plies=4, n_rand_black=2, n_rand_white=2, weights=dev_w(xu.int_weights(5)))
    full, tot, summ = run(n, **kw)
    h = n // 2
    halves = [run(h, gid0=0, **kw), run(n - h, gid0=h, **kw)]

    def joined(parts):
        po = ops.Playout(n, full.t_max, torch.cat([p.black for p, _, _ in parts], 1),
                         torch.cat([p.white for p, _, _ in parts], 1), torch.cat([p.move for p, _, _ in parts], 1),
                         torch.cat([p.nplies for p, _, _ in parts]), torch.cat([p.final_black for p, _, _ in parts]),
                         torch.cat([p.final_white for p, _, _ in parts]))
        return po, sum(t for _, t, _ in parts), torch.cat([s for _, _, s in parts])

    for parts in (halves, None):
        if parts is None:                                          # the two halves at once, on two streams
            streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]
            torch.cuda.synchronize()
            parts = []
            for s, (g0, m) in zip(streams, ((0, h), (h, n - h))):
                with torch.cuda.stream(s):
                    parts.append(run(m, gid0=g0, **kw))
            torch.cuda.synchronize()
        po, t, s = joined(parts)
        assert_same_games(po, full, full.t_max)
        assert torch.equal(t, tot) and torch.equal(s, summ)


def test_learner_depth_option():
    from subproc_b200 import learner
    games = 4096
    a, b = learner.ProgressPositionMovesLearn(), learner.ProgressPositionMovesLearn()
    po_a, rows_a = a.self_play_iteration(games, seed=3, iteration=2, device=DEV)
    po_b, rows_b = b.self_play_iteration(games, seed=3, iteration=2, device=DEV, depth=1)
    assert torch.equal(ops.learn_accumulate(po_a), ops.learn_accumulate(po_b))
    assert rows_a == rows_b and a.params == b.params
    # two on-device iterations of depth-3 self-play = the same steps by hand
    c = learner.ProgressPositionMovesLearn()
    c.self_play_iterations_on_device(2, games, seed=4, random_plies=8, device=DEV, depth=3)
    w = torch.from_numpy(learner.ProgressPositionMovesLearn().weights_table()).to(DEV)
    acc = torch.zeros((4, ops.N_ACC), dtype=torch.int64, device=DEV)
    for it in range(2):
        po = ops.playout(games, seed=4, gid0=it * games, device=DEV, policy=S, depth=3, random_plies=8, weights=w)
        ops.learn_accumulate(po, acc=acc, lam=0.90)
        w, params, _ = ops.learn_refit(acc, w, clear=True)
    assert c.params == [int(v) for v in params.cpu().tolist()]
    greedy = learner.ProgressPositionMovesLearn()
    greedy.self_play_iterations_on_device(2, games, seed=4, random_plies=8, device=DEV)
    assert greedy.params != c.params                               # the searched games are other games


def test_arguments():
    w = dev_w(xu.default_weights())
    for depth in (None, 0, 13):
        with pytest.raises(ValueError):
            ops.playout(8, device=DEV, policy=S, weights=w, depth=depth)
        with pytest.raises(ValueError):
            ops.playout(8, device=DEV, policy=G, policy_white=S, weights=w, depth=3, depth_white=depth if depth else 0)
    po = ops.playout(0, device=DEV, policy=S, depth=3, weights=w)                 # an empty batch is a no-op
    assert po.nplies.numel() == 0
    # the C ABI on real buffers
    n = 64
    out = ops.playout(n, device=DEV)
    ws = torch.zeros(int(_lib.lib().othello_search_workspace_bytes()), dtype=torch.uint8, device=DEV)

    def call(**kw):
        a = _lib.PlayoutArgs()
        a.n_games, a.policy, a.policy_white, a.search_depth = n, S, -1, 3
        a.weights = ctypes.c_void_p(w.data_ptr())
        a.nplies, a.final_black, a.final_white = (ctypes.c_void_p(t.data_ptr()) for t in
                                                  (out.nplies, out.final_black, out.final_white))
        a.workspace, a.workspace_bytes = ctypes.c_void_p(ws.data_ptr()), ws.numel()
        for k, v in kw.items():
            setattr(a, k, v)
        rc = _lib.lib().othello_playout(ctypes.byref(a), ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream))
        torch.cuda.synchronize()
        return rc

    assert call() == 0 and bool((out.nplies > 0).all())
    assert call(search_depth=0) == -1 and call(search_depth=13) == -1
    assert call(weights=None) == -1 and call(policy=3) == -1
    assert call(workspace=None) == -2 and call(workspace_bytes=ws.numel() - 1) == -2
    assert call(n_games=0, policy=3) == 0
