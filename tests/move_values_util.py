"""Helpers of the move-value tests: the host build of the rows the kernels write (tests/move_values_host.cpp ->
csrc/move_values.cuh), built once per process (tests/host_build.py), run over threads (ctypes releases the GIL); and
the row reductions the tests compare with othello_search / othello_solve."""
import ctypes
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

import host_build
import search_util as xu
from solve_util import _inputs, _p

SLOTS = 65
REFUSED = -128


def host_lib():
    return host_build.load("move_values_host.cpp")


def _split(n, run, threads=None):
    """run(lo, hi) over chunks of the n positions, on threads"""
    step = max(1, -(-n // (4 * (threads or os.cpu_count() or 1))))
    with ThreadPoolExecutor(threads or os.cpu_count() or 1) as ex:
        list(ex.map(lambda lo: run(lo, min(n, lo + step)), range(0, n, step)))


def host_search_moves(black, white, turn, weights, depth):
    """(values float32 [n][65], nodes uint64 [n][65]) of the host build"""
    b, w, t = _inputs(black, white, turn)
    n = b.size
    values, nodes = np.zeros((n, SLOTS), np.float32), np.zeros((n, SLOTS), np.uint64)
    wf = xu.weights40(weights)
    L = host_lib()
    _split(n, lambda lo, hi: L.mv_search_moves(_p(b[lo:]), _p(w[lo:]), _p(t[lo:]), _p(wf), ctypes.c_int(depth),
                                               _p(values[lo:]), _p(nodes[lo:]), ctypes.c_long(hi - lo)))
    return values, nodes


def host_solve_moves(black, white, turn):
    """(values int32 [n][65], nodes uint64 [n][65]) of the host build"""
    b, w, t = _inputs(black, white, turn)
    n = b.size
    values, nodes = np.zeros((n, SLOTS), np.int32), np.zeros((n, SLOTS), np.uint64)
    L = host_lib()
    _split(n, lambda lo, hi: L.mv_solve_moves(_p(b[lo:]), _p(w[lo:]), _p(t[lo:]), _p(values[lo:]), _p(nodes[lo:]),
                                              ctypes.c_long(hi - lo)))
    return values, nodes


def oracle_rows(b, w, t, weights, depth):
    """(float64 [n][65], the reference's moves) from tests/search_oracle.c: orc_search_children for the squares,
    orc_search for a must-pass root's column 64, NaN elsewhere"""
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        squares = list(ex.map(lambda i: xu.oracle_children(b[i], w[i], t[i], weights, depth), range(b.size)))
    v0, m0 = xu.oracle_search(b, w, t, weights, depth)
    return np.concatenate([np.array(squares), np.where(m0 == xu.PASS, v0, np.nan)[:, None]], axis=1), m0


def row_max_search(values):
    """(max float32 [n], lowest arg-max uint8 [n]) of the finite entries of each row; (NaN, 255) for a row without"""
    finite = ~np.isnan(values)
    v = np.where(finite, values, -np.inf)
    arg = np.argmax(v, axis=1)                          # the first maximum: the lowest index reaching it
    best = v[np.arange(values.shape[0]), arg]
    has = finite.any(axis=1)
    return np.where(has, best, np.nan).astype(np.float32), np.where(has, arg, 255).astype(np.uint8)


def row_max_solve(values):
    """(max int32 [n], lowest arg-max uint8 [n]) of the entries of each row that are not REFUSED; (REFUSED, 255) for
    a row without"""
    v = np.where(values == REFUSED, -1000, values)
    arg = np.argmax(v, axis=1)
    has = (values != REFUSED).any(axis=1)
    return (np.where(has, v[np.arange(values.shape[0]), arg], REFUSED).astype(np.int32),
            np.where(has, arg, 255).astype(np.uint8))


def legal_masks(oracle, b, w, t):
    """uint64 [n]: the legal moves of the side to move"""
    return np.asarray(oracle.puttables(b, w, t), np.uint64)


def legal_slots(legal):
    """bool [n][65]: which squares are legal (the pass column False)"""
    bits = (np.asarray(legal, np.uint64)[:, None] >> np.arange(64, dtype=np.uint64)[None, :]) & np.uint64(1)
    return np.concatenate([bits.astype(bool), np.zeros((bits.shape[0], 1), bool)], axis=1)
