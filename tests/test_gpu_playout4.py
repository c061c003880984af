"""The random playout kernel plays four games per thread (lane l, slot k of warp w: game 128 w + 32 k + l): batches
that leave slots, lanes and warps empty, games of one thread that start from different positions and colours, and
truncated trajectories, bit-exact against the oracle; the per-game summaries and the launch totals summed over the
four games of a thread."""
import numpy as np
import pytest
import torch

from subproc_b200 import ops
from gpu_util import DEV, dev_bits, dev_u8, host_bits, sample_positions
from test_gpu_playout import check_against_oracle

pytestmark = pytest.mark.gpu


def check_summary_and_totals(po, tot, sm, ref):
    nb = np.array([bin(int(v)).count("1") for v in ref['final_black']])
    nw = np.array([bin(int(v)).count("1") for v in ref['final_white']])
    want = [int(ref['nplies'].sum()), int((nb - nw).sum()), int((nb > nw).sum()), int((nw > nb).sum())]
    assert tot.cpu().tolist() == want
    smv = sm.cpu().numpy().view(np.uint16)
    assert np.array_equal(smv & 0xff, np.minimum(ref['nplies'], 255))
    assert np.array_equal((smv >> 8).astype(np.uint8).view(np.int8), (nb - nw).astype(np.int8))


@pytest.mark.parametrize("n", [1, 31, 33, 127, 129, 513])
def test_ragged_batches_bit_exact(oracle, n):
    tot = torch.zeros(4, dtype=torch.int64, device=DEV)
    sm = torch.zeros(n, dtype=torch.int16, device=DEV)
    po = ops.playout(n, seed=23, gid0=5, device=DEV, totals=tot, summary=sm)
    ref = oracle.playout(23, 5, n)
    check_against_oracle(po, ref, n)
    check_summary_and_totals(po, tot, sm, ref)
    nt = ops.playout(n, seed=23, gid0=5, device=DEV, trajectory=False)
    assert np.array_equal(nt.nplies.cpu().numpy(), ref['nplies'])
    assert np.array_equal(host_bits(nt.final_black), ref['final_black'])


@pytest.mark.parametrize("n", [33, 129, 515])
def test_mixed_starts_and_turns_within_a_thread(oracle, n):
    """neighbouring slots of a thread get unrelated positions and colours; some slots get the standard opening"""
    b, w = sample_positions(oracle, 60, seed=43, stride=2)
    rng = np.random.RandomState(n)
    pick = rng.randint(0, b.size, size=n)
    b, w = b[pick].copy(), w[pick].copy()
    std = rng.rand(n) < 0.3
    b[std], w[std] = oracle.START_BLACK, oracle.START_WHITE
    turn = rng.randint(1, 3, size=n).astype(np.uint8)
    tot = torch.zeros(4, dtype=torch.int64, device=DEV)
    sm = torch.zeros(n, dtype=torch.int16, device=DEV)
    po = ops.playout(n, seed=31, gid0=11, device=DEV, black0=dev_bits(b), white0=dev_bits(w), turn0=dev_u8(turn),
                     totals=tot, summary=sm)
    ref = oracle.playout(31, 11, n, black0=b, white0=w, turn0=turn)
    check_against_oracle(po, ref, n)
    check_summary_and_totals(po, tot, sm, ref)
    # the same positions with Black to move everywhere (no per-game turns)
    po = ops.playout(n, seed=31, gid0=11, device=DEV, black0=dev_bits(b), white0=dev_bits(w))
    check_against_oracle(po, oracle.playout(31, 11, n, black0=b, white0=w), n)


@pytest.mark.parametrize("t_max", [1, 5, 9, 37])
def test_truncated_trajectories(oracle, t_max):
    n = 129
    po = ops.playout(n, seed=4, gid0=0, device=DEV, t_max=t_max)
    check_against_oracle(po, oracle.playout(4, 0, n, t_max=t_max), n)
    b, w = sample_positions(oracle, 20, seed=44, stride=5)
    b, w = b[:n], w[:n]
    turn = (np.arange(b.size) % 3 == 0).astype(np.uint8) + 1
    po = ops.playout(b.size, seed=4, gid0=0, device=DEV, t_max=t_max, black0=dev_bits(b), white0=dev_bits(w),
                     turn0=dev_u8(turn))
    check_against_oracle(po, oracle.playout(4, 0, b.size, t_max=t_max, black0=b, white0=w, turn0=turn), b.size)
