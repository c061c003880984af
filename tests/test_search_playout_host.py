"""Search self-play without a GPU: the referee of tests/test_gpu_search_playout.py is checked against the oracle's own
greedy games (a greedy engine is a search engine of depth 1), and othello_playout refuses bad search arguments before
it touches a device."""
import ctypes

import numpy as np
import pytest

import search_playout_util as pu
import search_util as xu


@pytest.mark.parametrize("config", [
    dict(random_plies=0),
    dict(random_plies=6, n_rand_black=3, n_rand_white=5),
    dict(random_plies=2, n_rand_black=4, policy_white=pu.RANDOM),
    dict(random_plies=0, n_rand_white=2, policy=pu.RANDOM, policy_white=pu.SEARCH),
])
def test_referee_at_depth_1_is_the_oracle_greedy_game(oracle, config):
    n, seed, gid0 = 96, 41, 1000
    w1, w2 = xu.int_weights(51), xu.int_weights(52)
    ref = pu.referee(oracle, n, seed=seed, gid0=gid0, depth=1, weights=w1, weights_white=w2, **config)
    greedy = {pu.SEARCH: oracle.POLICY_GREEDY, pu.RANDOM: oracle.POLICY_RANDOM}
    pol = greedy[config.get("policy", pu.SEARCH)]
    pol_w = greedy[config.get("policy_white", config.get("policy", pu.SEARCH))]
    want = oracle.playout(seed, gid0, n, policy=pol, policy_white=pol_w, random_plies=config["random_plies"],
                          n_rand_black=config.get("n_rand_black", 0), n_rand_white=config.get("n_rand_white", 0),
                          weights=w1, weights_white=w2)
    for k in ("black", "white", "move", "nplies", "final_black", "final_white"):
        assert np.array_equal(ref[k], want[k]), k
    assert ref["totals"][0] == int(want["nplies"].sum())
    assert len(ref["searched"]) > 10 * n                          # most plies went to the search


def _args(**kw):
    """othello_playout_args of a 4-game search batch with dummy (never dereferenced) pointers"""
    from subproc_b200 import _lib
    a = _lib.PlayoutArgs()
    a.n_games, a.policy, a.policy_white, a.search_depth = 4, 2, -1, 3
    dummy = ctypes.c_void_p(4096)
    a.weights, a.nplies, a.final_black, a.final_white = dummy, dummy, dummy, dummy
    a.workspace, a.workspace_bytes = dummy, 1 << 20
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_c_abi_refuses_bad_search_arguments_without_a_device():
    from subproc_b200 import _lib
    L = _lib.lib()
    play = lambda **kw: L.othello_playout(ctypes.byref(_args(**kw)), None)
    E_INVALID, E_WORKSPACE = -1, -2
    for depth in (0, 13, -1):
        assert play(search_depth=depth) == E_INVALID
    assert play(policy=3) == E_INVALID and play(policy_white=3) == E_INVALID and play(policy_white=-2) == E_INVALID
    assert play(weights=None) == E_INVALID                            # Black searches without a table
    assert play(policy=0, policy_white=2, search_depth=0, search_depth_white=0) == E_INVALID   # White's depth
    assert play(policy=0, policy_white=2, weights=None) == E_INVALID
    assert play(policy=1, policy_white=2, search_depth=0, search_depth_white=13) == E_INVALID
    assert play(workspace=None) == E_WORKSPACE
    assert play(workspace_bytes=L.othello_search_workspace_bytes() - 1) == E_WORKSPACE
    assert play(n_games=0, policy=3) == 0                             # an empty batch is a no-op
    assert L.othello_abi_version() == 6
