"""The tuned rules primitives (csrc/fastboard.cuh: all-left floods on the board and its 180-degree
rotation, carry-propagation rows and rays) compiled for the HOST and compared with the oracle.
Same source as the kernels, so algorithmic slips are caught on the CPU box."""
import ctypes

import numpy as np
import pytest

import host_build


@pytest.fixture(scope="module")
def fb():
    return host_build.load("fastboard_host.cpp")


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def positions(oracle, n_games, seed):
    r = oracle.playout(seed, 0, n_games)
    bs, ws = [], []
    for g in range(n_games):
        n = int(r['nplies'][g])
        bs.append(r['black'][:n + 1, g])
        ws.append(r['white'][:n + 1, g])
    return np.concatenate(bs), np.concatenate(ws)


def test_fast_legal_and_flips_match_oracle(fb, oracle):
    b, w = positions(oracle, 500, 51)
    rng = np.random.RandomState(1)
    n = b.size
    occ = rng.randint(0, 2 ** 62, size=20000).astype(np.uint64) | (rng.randint(0, 4, size=20000).astype(np.uint64) << np.uint64(62))
    col = rng.randint(0, 2 ** 62, size=20000).astype(np.uint64) | (rng.randint(0, 4, size=20000).astype(np.uint64) << np.uint64(62))
    b = np.ascontiguousarray(np.concatenate([b, occ & col]))
    w = np.ascontiguousarray(np.concatenate([w, occ & ~col]))
    n = b.size
    out = np.zeros(n, dtype=np.uint64)
    for own, opp, piece in ((b, w, 1), (w, b, 2)):
        fb.fb_legal(P(own), P(opp), P(out), ctypes.c_long(n))
        assert np.array_equal(out, oracle.puttables(b, w, piece))
        sq = rng.randint(0, 64, size=n).astype(np.uint8)
        legal = oracle.puttables(b, w, piece)
        for i in range(0, n, 3):                         # bias a third of the squares towards legal moves
            if legal[i]:
                bits = [s for s in range(64) if (int(legal[i]) >> s) & 1]
                sq[i] = bits[rng.randint(len(bits))]
        fb.fb_flips(P(own), P(opp), P(sq), P(out), ctypes.c_long(n))
        _, _, want, _ = oracle.put(b, w, piece, sq)
        assert np.array_equal(out, want)
        fb.fb_flips_rowlut(P(own), P(opp), P(sq), P(out), ctypes.c_long(n))      # horizontal rays by rank look-up
        assert np.array_equal(out, want)
        fb.fb_flips_lut(P(own), P(opp), P(sq), P(out), ctypes.c_long(n))         # all four lines by look-up
        assert np.array_equal(out, want)
        fb.fb_flips_lut_line(P(own), P(opp), P(sq), P(out), ctypes.c_long(own.size))    # ... diagonal masks by diagonal number (greedy kernel)
        assert np.array_equal(out, want)


def test_constructed_lines_every_direction_square_and_run_length(fb, oracle):
    """runs of 0..7 opponent discs from every square in every direction, closed / open / into the edge"""
    import line_cases
    own, opp, sq = line_cases.build()
    n = own.size
    assert n > 5000
    out = np.zeros(n, dtype=np.uint64)
    fb.fb_legal(P(own), P(opp), P(out), ctypes.c_long(n))
    assert np.array_equal(out, oracle.puttables(own, opp, 1))
    fb.fb_flips(P(own), P(opp), P(sq), P(out), ctypes.c_long(n))
    _, _, want, ret = oracle.put(own, opp, 1, sq)
    assert np.array_equal(out, want)
    fb.fb_flips_rowlut(P(own), P(opp), P(sq), P(out), ctypes.c_long(n))
    assert np.array_equal(out, want)
    fb.fb_flips_lut(P(own), P(opp), P(sq), P(out), ctypes.c_long(n))
    assert np.array_equal(out, want)
    fb.fb_flips_lut_line(P(own), P(opp), P(sq), P(out), ctypes.c_long(own.size))    # ... diagonal masks by diagonal number (greedy kernel)
    assert np.array_equal(out, want)
    assert (ret >= 6).sum() > 50 and (ret == 0).sum() > 1000          # six-disc runs and dead rays are both present


def test_mobility_of_both_colours_in_one_pass(fb, oracle):
    """obf::mobility_both (shared conversions, popcount in the interleaved layout) == popcount of puttables()"""
    b, w = positions(oracle, 300, 52)
    rng = np.random.RandomState(3)
    occ = rng.randint(0, 2 ** 62, size=5000).astype(np.uint64) | (rng.randint(0, 4, size=5000).astype(np.uint64) << np.uint64(62))
    col = rng.randint(0, 2 ** 62, size=5000).astype(np.uint64) | (rng.randint(0, 4, size=5000).astype(np.uint64) << np.uint64(62))
    b = np.ascontiguousarray(np.concatenate([b, occ & col]))
    w = np.ascontiguousarray(np.concatenate([w, occ & ~col]))
    n = b.size
    mb, mw = np.zeros(n, np.int32), np.zeros(n, np.int32)
    fb.fb_mobility_both(P(b), P(w), P(mb), P(mw), ctypes.c_long(n))
    pop = lambda a: np.array([bin(int(v)).count("1") for v in a], dtype=np.int32)
    assert np.array_equal(mb, pop(oracle.puttables(b, w, 1))) and np.array_equal(mw, pop(oracle.puttables(b, w, 2)))
    # obf::mobility (one colour, mask never converted back to the standard layout): what counts() / the evaluation use
    m1, m2 = np.zeros(n, np.int32), np.zeros(n, np.int32)
    fb.fb_mobility(P(b), P(w), P(m1), ctypes.c_long(n))
    fb.fb_mobility(P(w), P(b), P(m2), ctypes.c_long(n))
    assert np.array_equal(m1, mb) and np.array_equal(m2, mw)


def test_child_mobility_from_the_prepared_parent(fb, oracle):
    """obf::child_mobility (successor built in the interleaved layout from the parent + the placed discs) ==
    the mover's n_puttable_for after put() in the oracle"""
    b, w = positions(oracle, 200, 53)
    n = b.size
    rng = np.random.RandomState(4)
    for own, opp, piece in ((b, w, 1), (w, b, 2)):
        legal = oracle.puttables(b, w, piece)
        sq = rng.randint(0, 64, size=n).astype(np.uint8)
        for i in range(n):
            if legal[i]:
                bits = [s for s in range(64) if (int(legal[i]) >> s) & 1]
                sq[i] = bits[rng.randint(len(bits))]
        got = np.zeros(n, np.int32)
        fb.fb_child_mobility(P(own), P(opp), P(sq), P(got), ctypes.c_long(n))
        nb, nw, flips, _ = oracle.put(b, w, piece, sq)
        after = oracle.puttables(nb, nw, piece)
        want = np.array([bin(int(v)).count("1") if f else -1 for v, f in zip(after, flips)], dtype=np.int32)
        assert np.array_equal(got, want)


def test_rank_tables_every_rank_file_and_pattern(fb, oracle):
    """the rank look-up of the horizontal rays (obf::row_flips): every rank, every file, all 3^7 fillings of the other
    seven squares of the rank, other ranks filled at random (they must not matter to the two horizontal rays, and the
    remaining six rays still go through the carry chains)"""
    rng = np.random.RandomState(7)
    pats = np.array(np.meshgrid(*[[0, 1, 2]] * 7, indexing='ij')).reshape(7, -1).T       # 2187 x 7
    own_l, opp_l, sq_l = [], [], []
    for y in range(8):
        for x in range(8):
            cols = [c for c in range(8) if c != x]
            o = np.zeros(len(pats), dtype=np.uint64)
            p = np.zeros(len(pats), dtype=np.uint64)
            for j, c in enumerate(cols):
                o |= (pats[:, j] == 1).astype(np.uint64) << np.uint64(8 * y + c)
                p |= (pats[:, j] == 2).astype(np.uint64) << np.uint64(8 * y + c)
            noise_occ = rng.randint(0, 2 ** 62, size=len(pats)).astype(np.uint64) << np.uint64(2)
            noise_col = rng.randint(0, 2 ** 62, size=len(pats)).astype(np.uint64) << np.uint64(2)
            keep = ~(np.uint64(0xff) << np.uint64(8 * y))
            own_l.append(o | (noise_occ & noise_col & keep))
            opp_l.append(p | (noise_occ & ~noise_col & keep))
            sq_l.append(np.full(len(pats), 8 * y + x, dtype=np.uint8))
    own = np.ascontiguousarray(np.concatenate(own_l)); opp = np.ascontiguousarray(np.concatenate(opp_l))
    sq = np.ascontiguousarray(np.concatenate(sq_l))
    out = np.zeros(own.size, dtype=np.uint64)
    fb.fb_flips_rowlut(P(own), P(opp), P(sq), P(out), ctypes.c_long(own.size))
    _, _, want, _ = oracle.put(own, opp, 1, sq)
    assert own.size == 64 * 2187 and np.array_equal(out, want)
    fb.fb_flips_lut(P(own), P(opp), P(sq), P(out), ctypes.c_long(own.size))
    assert np.array_equal(out, want)
    fb.fb_flips_lut_line(P(own), P(opp), P(sq), P(out), ctypes.c_long(own.size))    # ... diagonal masks by diagonal number (greedy kernel)
    assert np.array_equal(out, want)


def test_kth_set_bit_table(fb):
    """[byte][k] -> position of the k-th set bit (the last step of obf::kth_set_bit in the playout kernel)"""
    for v in range(256):
        bits = [i for i in range(8) if (v >> i) & 1]
        for k, want in enumerate(bits):
            assert fb.fb_kth_table(v, k) == want


def test_line_tables_every_square_line_and_pattern(fb, oracle):
    """put() by line look-ups (obf::flips_lut, what the game kernels run): for every square and each of the four
    lines through it (rank, file, both diagonals) all 3^(L-1) fillings of the other squares of the line, the rest of
    the board filled at random -- the gathers (PRMT / multiplies), both tables and the scatters against the oracle"""
    rng = np.random.RandomState(11)
    own_l, opp_l, sq_l = [], [], []
    for s in range(64):
        x, y = s & 7, s >> 3
        for dx, dy in ((1, 0), (0, 1), (1, 1), (1, -1)):
            line = [(x + k * dx) + 8 * (y + k * dy) for k in range(-7, 8)
                    if k != 0 and 0 <= x + k * dx < 8 and 0 <= y + k * dy < 8]
            if not line:                                       # the one-square diagonal of a corner
                continue
            pats = np.array(np.meshgrid(*[[0, 1, 2]] * len(line), indexing='ij')).reshape(len(line), -1).T
            o = np.zeros(len(pats), dtype=np.uint64)
            p = np.zeros(len(pats), dtype=np.uint64)
            keep = ~np.uint64(1 << s)
            for j, c in enumerate(line):
                o |= (pats[:, j] == 1).astype(np.uint64) << np.uint64(c)
                p |= (pats[:, j] == 2).astype(np.uint64) << np.uint64(c)
                keep &= ~np.uint64(1 << c)
            occ = rng.randint(0, 2 ** 62, size=len(pats)).astype(np.uint64) << np.uint64(2) | rng.randint(0, 4, size=len(pats)).astype(np.uint64)
            col = rng.randint(0, 2 ** 62, size=len(pats)).astype(np.uint64) << np.uint64(2) | rng.randint(0, 4, size=len(pats)).astype(np.uint64)
            own_l.append(o | (occ & col & keep))
            opp_l.append(p | (occ & ~col & keep))
            sq_l.append(np.full(len(pats), s, dtype=np.uint8))
    own = np.ascontiguousarray(np.concatenate(own_l)); opp = np.ascontiguousarray(np.concatenate(opp_l))
    sq = np.ascontiguousarray(np.concatenate(sq_l))
    assert own.size > 300000 and not np.any(own & opp)
    out = np.zeros(own.size, dtype=np.uint64)
    fb.fb_flips_lut(P(own), P(opp), P(sq), P(out), ctypes.c_long(own.size))
    _, _, want, _ = oracle.put(own, opp, 1, sq)
    assert np.array_equal(out, want)
    out2 = np.zeros(own.size, dtype=np.uint64)
    fb.fb_flips_lut_line(P(own), P(opp), P(sq), P(out2), ctypes.c_long(own.size))    # diagonal masks by diagonal number
    assert np.array_equal(out2, want)
