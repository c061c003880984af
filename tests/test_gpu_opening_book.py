"""The random playout kernel's opening book (csrc/opening_book.cuh) on a B200: warps whose games all start from the
standard opening with Black to move take their first plies from the book; every game must still be the oracle's,
row for row, whatever the capacity, the start positions of the other lanes of the warp or the entry point."""
import ctypes

import numpy as np
import pytest

from subproc_b200 import _lib, ops
from gpu_util import DEV, dev_bits, dev_u8, host_bits, sample_positions

pytestmark = pytest.mark.gpu

# around both book depths worth building (6 and 8) and the longest game
T_MAX = [0, 1, 5, 6, 7, 8, 9, 20, 120]


def check(nplies, fb, fw, tb, tw, tm, ref, t_max):
    assert np.array_equal(nplies, ref["nplies"])
    assert np.array_equal(fb, ref["final_black"]) and np.array_equal(fw, ref["final_white"])
    if tb is None:
        return
    t_idx = np.arange(t_max + 1)[:, None]
    vp = t_idx <= np.minimum(nplies, t_max)[None, :]
    vm = t_idx[:-1] < np.minimum(nplies, t_max)[None, :]
    assert np.array_equal(tb[vp], ref["black"][vp]) and np.array_equal(tw[vp], ref["white"][vp])
    assert np.array_equal(tm[vm], ref["move"][vm])


def check_playout(po, ref):
    traj = po.black is not None
    check(po.nplies.cpu().numpy(), host_bits(po.final_black), host_bits(po.final_white),
          host_bits(po.black) if traj else None, host_bits(po.white) if traj else None,
          po.move.cpu().numpy() if traj else None, ref, po.t_max)


@pytest.mark.parametrize("t_max", T_MAX)
def test_standard_opening_every_capacity(oracle, t_max):
    n = 1000 + 13                                           # the last warp is ragged
    po = ops.playout(n, seed=11, gid0=45, device=DEV, t_max=t_max)
    check_playout(po, oracle.playout(11, 45, n, t_max=t_max))


@pytest.mark.parametrize("seed,gid0", [(0, 1), (3, 33), (2 ** 40 + 5, 1000003), (2 ** 64 - 1, 2 ** 63 - 7)])
def test_standard_opening_seeds_and_game_ids(oracle, seed, gid0):
    n = 777
    po = ops.playout(n, seed=seed, gid0=gid0, device=DEV)
    check_playout(po, oracle.playout(seed, gid0, n))
    bare = ops.playout(n, seed=seed, gid0=gid0, device=DEV, trajectory=False)           # no trajectory at all
    check_playout(bare, oracle.playout(seed, gid0, n, trajectory=False))


def mixed_starts(oracle):
    """warp 0: all standard, Black to move; warp 1: one lane with White to move on the standard position; warp 2:
    one custom start; warp 3: custom starts only; warp 4 (ragged): standard"""
    b, w = sample_positions(oracle, 8, seed=71)
    n = 4 * 32 + 19
    b0 = np.full(n, oracle.START_BLACK, np.uint64)
    w0 = np.full(n, oracle.START_WHITE, np.uint64)
    turn = np.full(n, oracle.BLACK, np.uint8)
    turn[32 + 17] = oracle.WHITE
    b0[64 + 5], w0[64 + 5] = b[40], w[40]
    b0[96:128], w0[96:128] = b[100:132], w[100:132]
    turn[96:128] = np.arange(32) % 2 + 1
    return n, b0, w0, turn


@pytest.mark.parametrize("t_max", [7, 120])
def test_warps_that_mix_standard_and_other_starts(oracle, t_max):
    n, b0, w0, turn = mixed_starts(oracle)
    po = ops.playout(n, seed=13, gid0=3, device=DEV, black0=dev_bits(b0), white0=dev_bits(w0), turn0=dev_u8(turn),
                     t_max=t_max)
    check_playout(po, oracle.playout(13, 3, n, black0=b0, white0=w0, turn0=turn, t_max=t_max))
    bare = ops.playout(n, seed=13, gid0=3, device=DEV, black0=dev_bits(b0), white0=dev_bits(w0), turn0=dev_u8(turn),
                       trajectory=False)
    check_playout(bare, oracle.playout(13, 3, n, black0=b0, white0=w0, turn0=turn, trajectory=False))
    # the same starts with Black to move everywhere (no turn0): warp 1 now qualifies
    po = ops.playout(n, seed=14, gid0=3, device=DEV, black0=dev_bits(b0), white0=dev_bits(w0), t_max=t_max)
    check_playout(po, oracle.playout(14, 3, n, black0=b0, white0=w0, t_max=t_max))


def test_uploaded_standard_starts_through_the_host_api(oracle):
    L = _lib.lib()
    ctx = ctypes.c_void_p()
    assert L.othello_ctx_create(0, ctypes.byref(ctx)) == 0
    try:
        n, t_max = 2000 + 5, 120
        b0 = np.full(n, oracle.START_BLACK, np.uint64)
        w0 = np.full(n, oracle.START_WHITE, np.uint64)
        tb, tw = np.zeros((t_max + 1, n), np.uint64), np.zeros((t_max + 1, n), np.uint64)
        tm = np.zeros((t_max, n), np.uint8)
        npl, fb, fw = np.zeros(n, np.int32), np.zeros(n, np.uint64), np.zeros(n, np.uint64)
        P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        assert L.othello_playout_host(ctx, 17, 1001, n, P(b0), P(w0), None, ops.POLICY_RANDOM, 0, 0, 0, None, -1, None,
                                      t_max, P(tb), P(tw), P(tm), P(npl), P(fb), P(fw)) == 0
        check(npl, fb, fw, tb, tw, tm, oracle.playout(17, 1001, n, black0=b0, white0=w0, t_max=t_max), t_max)
    finally:
        L.othello_ctx_destroy(ctx)
