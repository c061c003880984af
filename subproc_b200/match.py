"""The reference's match entry point (subproc.py:7-39) over the GPU game runner.

``do_match(conf)`` reads the same flat config keys (config.py:4-16 produces ``<section>_<option>``):
``proc_a_path`` / ``proc_b_path`` -- here engine specs instead of shell commands: ``random``,
``greedy`` (default_value() weights), ``greedy:<38-byte parameter file>``, ``search<D>`` (a D-ply alpha-beta search on
the default_value() weights) or ``search<D>:<parameter file>`` -- plus
``proc_n_rand_hands_for_a/b``, ``proc_debug``, ``proc_randomize_black_white`` and the recorder plugin
``game_recorder_from`` / ``game_recorder_class``.  Returns what play_a_game returns.
"""
import random

from . import paramgen, parameter
from .game_runner import GameRunner, Engine


def get_game_recorder(conf):                             # subproc.py:7-12
    mod = __import__(conf['game_recorder_from'], fromlist=[conf['game_recorder_class']])
    obj = getattr(mod, conf['game_recorder_class'])()
    obj.configure('', '', conf)
    return obj


def engine_from_spec(spec):
    P = parameter.ProgressPositionMovesParameter()
    if spec == 'random':
        return Engine('random')
    if spec == 'greedy':
        return Engine('greedy', P.weights_table())
    if spec.startswith('greedy:'):
        return Engine('greedy', P.weights_table(paramgen.read_data(spec.split(':', 1)[1])))
    kind, _, path = spec.partition(':')
    if kind.startswith('search') and kind[6:].isdigit():
        table = P.weights_table(paramgen.read_data(path)) if path else P.weights_table()
        return Engine('search', table, depth=int(kind[6:]))
    raise ValueError("unknown engine spec %r (expected random | greedy | greedy:<param file> | search<depth> | "
                     "search<depth>:<param file>)" % spec)


def do_match(conf, seed=0, device=None, recorder=None):
    """One match as configured (the job of subproc.py:15-39): engines and substitution budgets per side,
    optional colour swap, recorder plugin opened as a context manager, one game played."""
    sides = [(engine_from_spec(conf['proc_%s_path' % k]), int(conf.get('proc_n_rand_hands_for_%s' % k, 0)))
             for k in ('a', 'b')]
    if conf.get('proc_randomize_black_white', 0) == 1 and random.randrange(2) == 1:
        sides.reverse()                                   # "... and swapped black and white"
    (black, n_black), (white, n_white) = sides
    with (recorder if recorder is not None else get_game_recorder(conf)) as recorder:
        runner = GameRunner(black, white, recorder, conf.get('proc_debug', 0) == 1, n_black, n_white,
                            device=device, seed=seed)
        return runner.play_a_game()
