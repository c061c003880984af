"""The rank-sliced move generator of four boards at once (obf::legal_moves4 in csrc/fastboard.cuh, what the random
playout kernel runs) compiled for the HOST and compared with the oracle and with the one-board generator."""
import ctypes

import numpy as np
import pytest

import host_build


@pytest.fixture(scope="module")
def fb():
    return host_build.load("legal4_host.cpp")


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def pad4(*arrays):
    n = (arrays[0].size + 3) // 4 * 4
    return [np.ascontiguousarray(np.concatenate([a, np.zeros(n - a.size, a.dtype)])) for a in arrays]


def check(fb, oracle, b, w, rots=(0, 1, 2, 3)):
    """both colours, every position in every byte slot, against the oracle and obf::legal_moves"""
    b, w = pad4(b, w)
    n = b.size
    out, one = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
    for own, opp, piece in ((b, w, 1), (w, b, 2)):
        want = oracle.puttables(b, w, piece)
        fb.fb_legal(P(own), P(opp), P(one), ctypes.c_long(n))
        assert np.array_equal(one, want)
        for rot in rots:
            out[:] = 0
            fb.fb_legal4(P(own), P(opp), P(out), ctypes.c_long(n), ctypes.c_int(rot))
            assert np.array_equal(out, want), rot


def random_boards(rng, n):
    occ = rng.randint(0, 2 ** 62, size=n).astype(np.uint64) | (rng.randint(0, 4, size=n).astype(np.uint64) << np.uint64(62))
    col = rng.randint(0, 2 ** 62, size=n).astype(np.uint64) | (rng.randint(0, 4, size=n).astype(np.uint64) << np.uint64(62))
    return occ & col, occ & ~col


def test_sliced_layout_round_trip(fb):
    rng = np.random.RandomState(5)
    v = np.ascontiguousarray(rng.randint(0, 2 ** 63, size=64).astype(np.uint64) * np.uint64(3))
    out = np.zeros(64, np.uint64)
    words = np.zeros(128, np.uint32)
    fb.fb_sliced_round_trip(P(v), P(out), P(words), ctypes.c_long(64))
    assert np.array_equal(out, v)
    for i in range(0, 64, 4):                      # word r of a group: rank r of its four boards, board j in byte j
        for r in range(8):
            for j in range(4):
                assert (int(words[2 * i + r]) >> (8 * j)) & 0xff == (int(v[i + j]) >> (8 * r)) & 0xff


def test_played_and_random_positions(fb, oracle):
    r = oracle.playout(61, 0, 400)
    bs = [r['black'][:int(r['nplies'][g]) + 1, g] for g in range(400)]
    ws = [r['white'][:int(r['nplies'][g]) + 1, g] for g in range(400)]
    rb, rw = random_boards(np.random.RandomState(2), 40000)
    b, w = np.concatenate(bs + [rb]), np.concatenate(ws + [rw])
    # neighbours in a call are unrelated positions: shuffle so that every call mixes phases and games
    perm = np.random.RandomState(3).permutation(b.size)
    check(fb, oracle, b[perm], w[perm])


def test_constructed_lines_in_every_byte_slot(fb, oracle):
    """runs of 0..7 opponent discs from every square in every direction, closed / open / into the edge
    (tests/line_cases.py), each in all four byte slots, next to three other such positions"""
    import line_cases
    own, opp, _ = line_cases.build()
    assert own.size > 5000
    check(fb, oracle, own, opp)
    # the neighbours of a line position are dense boards: a run that leaked across a byte would change them
    rb, rw = random_boards(np.random.RandomState(9), own.size * 3)
    b = np.stack([own, rb[0::3], rb[1::3], rb[2::3]], axis=1).reshape(-1)
    w = np.stack([opp, rw[0::3], rw[1::3], rw[2::3]], axis=1).reshape(-1)
    check(fb, oracle, b, w)


def test_edge_files_and_full_ranks(fb, oracle):
    """boards whose files a / h and first / last ranks are full of discs: the bits a shift or a carry would move into
    the neighbouring game's byte"""
    rng = np.random.RandomState(13)
    edge = np.uint64(0x8181818181818181) | np.uint64(0xFF000000000000FF)
    b, w = random_boards(rng, 20000)
    col = rng.randint(0, 2 ** 62, size=20000).astype(np.uint64) * np.uint64(3)
    b = (b & ~edge) | (col & edge)
    w = (w & ~edge) | (~col & edge)
    check(fb, oracle, b, w)
