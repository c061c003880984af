"""The opening book of the random playout kernel (csrc/opening_book.cuh) compiled for the HOST and compared with the
oracle: the tree the kernel walks for the first plies of every game from the standard opening."""
import ctypes

import numpy as np
import pytest

import host_build

NODE = np.dtype([("black", "<u8"), ("white", "<u8"), ("first", "<u4"), ("info", "<u4"), ("pad", "<u4", (2,))])
# perft from the standard opening (BASELINE.md): move paths after 0..8 plies
PERFT = [1, 4, 12, 56, 244, 1396, 8200, 55092, 390216]


@pytest.fixture(scope="module")
def book():
    L = host_build.load("opening_book_host.cpp")
    L.ob_book_build.restype = ctypes.c_long
    L.ob_book_build.argtypes = [ctypes.c_int]
    L.ob_book_copy.argtypes = [ctypes.c_void_p]
    return L


def build(L, depth):
    n = L.ob_book_build(depth)
    assert n > 0
    nodes = np.zeros(n, dtype=NODE)
    L.ob_book_copy(nodes.ctypes.data_as(ctypes.c_void_p))
    return nodes


def test_tree_to_depth_8_against_the_oracle(book, oracle):
    nodes = build(book, 8)
    assert nodes.itemsize == 32 and len(nodes) == sum(PERFT)
    n = (nodes["info"] & 0xff).astype(np.int64)
    move = ((nodes["info"] >> 8) & 0xff).astype(np.uint8)
    first = nodes["first"].astype(np.int64)
    assert nodes["black"][0] == oracle.START_BLACK and nodes["white"][0] == oracle.START_WHITE
    begin = 0
    for d, count in enumerate(PERFT):
        end = begin + count
        lvl = slice(begin, end)
        if d == len(PERFT) - 1:
            assert end == len(nodes) and not n[lvl].any()          # the last ply: no links
            break
        # breadth first, children contiguous: the next level follows this one, node after node
        assert first[begin] == end and np.array_equal(first[begin + 1:end], first[begin:end - 1] + n[begin:end - 1])
        assert first[end - 1] + n[end - 1] == end + PERFT[d + 1]
        piece = oracle.BLACK if d % 2 == 0 else oracle.WHITE           # no pass above the last ply
        legal = oracle.puttables(nodes["black"][lvl], nodes["white"][lvl], piece)
        assert (legal != 0).all()                                      # every internal node has a move
        assert np.array_equal(n[lvl], np.bitwise_count(legal))
        # child c of parent p: the k-th legal move of p in ascending square order, and the oracle's put() result
        parent = np.repeat(np.arange(begin, end), n[lvl])
        child = np.arange(end, end + PERFT[d + 1])
        k = child - first[parent]
        mv = move[child]
        lp = legal[parent - begin]
        assert ((lp >> mv.astype(np.uint64)) & np.uint64(1)).all()
        below = lp & ((np.uint64(1) << mv.astype(np.uint64)) - np.uint64(1))
        assert np.array_equal(np.bitwise_count(below).astype(np.int64), k)
        nb, nw, flips, ret = oracle.put(nodes["black"][parent], nodes["white"][parent], piece, mv)
        assert (ret > 0).all()
        assert np.array_equal(nodes["black"][child], nb) and np.array_equal(nodes["white"][child], nw)
        begin = end


def test_builder_refuses_a_tree_with_a_pass(book):
    """24 positions after eight plies have no move for Black: a ninth book ply would need a pass"""
    assert book.ob_book_build(9) == -1

