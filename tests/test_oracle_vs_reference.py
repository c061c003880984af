"""The oracle against the reference.  The two game tests play fresh games on the reference's own board.py and run
only where its sources are reachable (oracle/_ref, see oracle/build_ref.py); without them the stored reference games
of tests/test_oracle_golden.py are the pin.  The evaluation test uses the reference's counts() stored with the golden
games and runs everywhere.
"""
import numpy as np
import pytest

from oracle import refshim
from oracle import make_golden as mg

live = pytest.mark.skipif(not refshim.available(), reason="needs the original project's sources (oracle/_ref, see "
                          "oracle/build_ref.py), which are not part of the repository")


@live
def test_random_games_against_live_reference(oracle):
    ns = refshim.load()
    rows = ns.ppml.ProgressPositionMovesParameter().default_value()
    for gid in range(100, 112):
        g = mg.play_game(ns, 11, gid, 0, 0, 0, 0, rows, record_features=True)
        pos = g['positions']
        b = np.array([int(p['b'], 16) for p in pos], dtype=np.uint64)
        w = np.array([int(p['w'], 16) for p in pos], dtype=np.uint64)
        assert [int(v) for v in oracle.puttables(b, w, 1)] == [int(p['legal_b'], 16) for p in pos]
        assert [int(v) for v in oracle.puttables(b, w, 2)] == [int(p['legal_w'], 16) for p in pos]
        assert oracle.features(b, w, 1).tolist() == [p['feat_O'] for p in pos]
        assert oracle.features(b, w, 2).tolist() == [p['feat_X'] for p in pos]
        r = oracle.playout(11, gid, 1)
        assert r['move'][:len(g['plies']), 0].tolist() == [p['move'] for p in g['plies']]


@live
def test_greedy_games_against_live_reference(oracle):
    ns = refshim.load()
    rows = ns.ppml.ProgressPositionMovesParameter().default_value()
    for gid in range(3):
        g = mg.play_game(ns, 12, gid, 1, 6, 0, 0, rows, record_features=False)
        r = oracle.playout(12, gid, 1, policy=1, random_plies=6)
        assert r['move'][:len(g['plies']), 0].tolist() == [p['move'] for p in g['plies']]
        assert int(r['nplies'][0]) == len(g['plies'])


def test_eval_against_counts_dot(oracle, golden_games):
    """the oracle's linear form against the dot product of the reference's own counts() of every position of the
    golden games that carry them (recorded by oracle/make_golden.py as feat_O / feat_X)"""
    rng = np.random.RandomState(3)
    w = np.concatenate([rng.uniform(-2, 2, size=(4, 9)), rng.uniform(-1, 1, size=(4, 1))], axis=1)
    checked = 0
    for g in golden_games:
        pos = g['positions']
        if 'feat_O' not in pos[0]:
            continue
        b = np.array([int(p['b'], 16) for p in pos], dtype=np.uint64)
        ww = np.array([int(p['w'], 16) for p in pos], dtype=np.uint64)
        for key, colour in (('feat_O', 1), ('feat_X', 2)):
            got = oracle.evaluate(b, ww, colour, w)
            for p, v in zip(pos, got):
                f = p[key]
                row = 0 if f[0] <= 16 else 1 if f[0] <= 32 else 2 if f[0] <= 48 else 3
                want = float(np.dot(w[row, :9], np.array(f[1:], dtype=np.float64)) + w[row, 9])
                assert abs(float(v) - want) <= 1e-12 * max(1.0, abs(want))
                checked += 1
    assert checked >= 900
