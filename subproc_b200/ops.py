"""Batched device operations: torch tensors in, hand-written sm_100a kernels through the C ABI.

torch is plumbing here (device memory, streams); every function below is one launch of a kernel
in subproc_b200/csrc through include/othello_b200.h.  Bitboards are ``torch.int64`` tensors
holding the uint64 bit pattern (bit s = x + 8*y, board.py:79); colours / moves are ``torch.uint8``.

There is no CPU path: tensors must live on a CUDA device and the library must be built.
"""
import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib

EMPTY, BLACK, WHITE = 0, 1, 2                    # board.py:3-7
PASS = 64                                        # 'ps' / 'PS' (board.py:194)
START_BLACK = 0x0000000810000000                 # board.py:25
START_WHITE = 0x0000001008000000                 # board.py:24
POLICY_RANDOM, POLICY_GREEDY, POLICY_SEARCH = 0, 1, 2
F_MUST_PASS, F_GAME_OVER = 1, 2
T_MAX_DEFAULT = 120                              # 60 moves + 60 interleaved passes

# square-class masks a..h (parameter_progress_position_moves_learn.py:9-16)
CLASS_MASKS = (0x8100000000000081, 0x4281000000008142, 0x0042000000004200, 0x2400810000810024,
               0x1800008181000018, 0x003C424242423C00, 0x0000240000240000, 0x0000183C3C180000)
# disc-count shards of the four weight rows (progress_position_moves_learn.py:112-113)
PHASE_SHARDS = ((0, 16), (17, 32), (33, 48), (49, 64))


def signed64(v):
    """python int bit pattern (0..2**64-1) -> the int64 value torch stores."""
    v &= 0xFFFFFFFFFFFFFFFF
    return v - (1 << 64) if v >= (1 << 63) else v


def unsigned64(v):
    return int(v) & 0xFFFFFFFFFFFFFFFF


def bits_tensor(values, device):
    """iterable of python ints / numpy uint64 -> int64 CUDA tensor of bit patterns."""
    a = np.asarray(values, dtype=np.uint64).reshape(-1).view(np.int64)
    return torch.from_numpy(a.copy()).to(device)


def bits_numpy(t):
    """int64 tensor of bit patterns -> numpy uint64 (host)."""
    return t.detach().cpu().numpy().view(np.uint64)


def _req(t, dtype, n=None, name="tensor"):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor (no CPU path exists)" % name)
    if t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if n is not None and t.numel() != n:
        raise ValueError("%s must have %d elements, got %d" % (name, n, t.numel()))
    return ctypes.c_void_p(t.data_ptr())


def _opt(t, dtype, n, name):
    return None if t is None else _req(t, dtype, n, name)


def _stream(t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def legal(own, opp, out=None):
    """Board.puttables(piece) as masks (board.py:46-52): own = discs of ``piece``."""
    n = own.numel()
    out = torch.empty_like(own) if out is None else out
    with torch.cuda.device(own.device):
        _lib.check(_lib.lib().othello_legal(_req(own, torch.int64, n, "own"), _req(opp, torch.int64, n, "opp"),
                                            _req(out, torch.int64, n, "out"), n, _stream(own)), "othello_legal")
    return out


def flips(own, opp, square, out=None):
    """Board.put(piece, x, y) flip sets (board.py:161-174); 0 where put would return 0."""
    n = own.numel()
    out = torch.empty_like(own) if out is None else out
    with torch.cuda.device(own.device):
        _lib.check(_lib.lib().othello_flips(_req(own, torch.int64, n, "own"), _req(opp, torch.int64, n, "opp"),
                                            _req(square, torch.uint8, n, "square"), _req(out, torch.int64, n, "out"),
                                            n, _stream(own)), "othello_flips")
    return out


def step(black, white, turn, nturn, move, flips_out=None, ret=None, flags=None):
    """Board.put_s for the side to move, IN PLACE (board.py:192-209).  Returns (flips, ret, flags)."""
    n = black.numel()
    dev = black.device
    flips_out = torch.empty(n, dtype=torch.int64, device=dev) if flips_out is None else flips_out
    ret = torch.empty(n, dtype=torch.int32, device=dev) if ret is None else ret
    flags = torch.empty(n, dtype=torch.uint8, device=dev) if flags is None else flags
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().othello_step(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"),
            _req(turn, torch.uint8, n, "turn"), _req(nturn, torch.int32, n, "nturn"),
            _req(move, torch.uint8, n, "move"), _req(flips_out, torch.int64, n, "flips_out"),
            _req(ret, torch.int32, n, "ret"), _req(flags, torch.uint8, n, "flags"), n, _stream(black)), "othello_step")
    return flips_out, ret, flags


def counts(black, white):
    """[n][3] int32: n_black, n_white, n_empty (board.py:37-44)."""
    n = black.numel()
    out = torch.empty((n, 3), dtype=torch.int32, device=black.device)
    with torch.cuda.device(black.device):
        _lib.check(_lib.lib().othello_counts(_req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"),
                                             _req(out, torch.int32, 3 * n, "out"), n, _stream(black)), "othello_counts")
    return out


def mask_count(black, white, color, mask):
    """Board.mask_count(color, mask) (board.py:74-81), element-wise."""
    n = black.numel()
    out = torch.empty(n, dtype=torch.int32, device=black.device)
    with torch.cuda.device(black.device):
        _lib.check(_lib.lib().othello_mask_count(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"),
            _req(color, torch.uint8, n, "color"), _req(mask, torch.int64, n, "mask"),
            _req(out, torch.int32, n, "out"), n, _stream(black)), "othello_mask_count")
    return out


def serialize_boards(black, white):
    """uint8 [n][64]: Board.serialize_board() of every position (board.py:223-243)."""
    n = black.numel()
    out = torch.empty((n, 64), dtype=torch.uint8, device=black.device)
    with torch.cuda.device(black.device):
        _lib.check(_lib.lib().othello_serialize_boards(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"),
            _req(out, torch.uint8, 64 * n, "out"), n, _stream(black)), "othello_serialize_boards")
    return out


def deserialize_boards(chars):
    """uint8 [n][64] board strings -> (black, white) int64 [n] (Board.deserialize, board.py:253-262)."""
    n = chars.shape[0]
    black = torch.empty(n, dtype=torch.int64, device=chars.device)
    white = torch.empty(n, dtype=torch.int64, device=chars.device)
    with torch.cuda.device(chars.device):
        _lib.check(_lib.lib().othello_deserialize_boards(
            _req(chars, torch.uint8, 64 * n, "chars"), _req(black, torch.int64, n, "black"),
            _req(white, torch.int64, n, "white"), n, _stream(chars)), "othello_deserialize_boards")
    return black, white


def features(black, white, side):
    """[n][10] int32 = counts(a_book, side) (parameter_progress_position_moves_learn.py:5-17)."""
    n = black.numel()
    out = torch.empty((n, 10), dtype=torch.int32, device=black.device)
    with torch.cuda.device(black.device):
        _lib.check(_lib.lib().othello_features(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"),
            _req(side, torch.uint8, n, "side"), _req(out, torch.int32, 10 * n, "out"), n, _stream(black)),
            "othello_features")
    return out


def weights_tensor(rows, device, intercepts=None):
    """4 rows x 9 weights (default_value() layout) [+ 4 intercepts] -> float32 [4][10] device tensor."""
    w = np.zeros((4, 10), dtype=np.float32)
    w[:, :9] = np.asarray(rows, dtype=np.float64).reshape(4, 9)
    if intercepts is not None:
        w[:, 9] = np.asarray(intercepts, dtype=np.float64).reshape(4)
    return torch.from_numpy(w).to(device)


def evaluate(black, white, side, weights):
    """float32 [n]: weights[phase] . (mobility, a..h) + weights[phase][9] for colour ``side``."""
    n = black.numel()
    out = torch.empty(n, dtype=torch.float32, device=black.device)
    with torch.cuda.device(black.device):
        _lib.check(_lib.lib().othello_eval(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"),
            _req(side, torch.uint8, n, "side"), _req(weights, torch.float32, 40, "weights"),
            _req(out, torch.float32, n, "out"), n, _stream(black)), "othello_eval")
    return out


@dataclass
class Playout:
    """Result of ``playout``: SoA trajectories [t][game] in HBM plus per-game results."""
    n_games: int
    t_max: int
    black: torch.Tensor          # int64 [t_max+1][n] position before ply t (None when trajectory=False)
    white: torch.Tensor
    move: torch.Tensor           # uint8 [t_max][n]; entries at t >= nplies[g] are unspecified
    nplies: torch.Tensor         # int32 [n] plies incl. passes = nturn of the terminal position
    final_black: torch.Tensor    # int64 [n]
    final_white: torch.Tensor

    def final_counts(self):
        return counts(self.final_black, self.final_white)

    def total_positions(self):
        """number of legal-gen+step position-steps executed (= plies played)."""
        return int(self.nplies.sum(dtype=torch.int64).item())


def playout(n_games, seed=0, gid0=0, device=None, black0=None, white0=None, turn0=None, policy=POLICY_RANDOM,
            random_plies=0, n_rand_black=0, n_rand_white=0, weights=None, t_max=T_MAX_DEFAULT, trajectory=True,
            out=None, policy_white=None, weights_white=None, totals=None, games_per_warp=0, summary=None, depth=None,
            depth_white=None):
    """GameRunner.play_a_game (game_runner.py:165-201) for n_games games in ONE kernel launch.

    Game g draws from the counter-based stream (seed, gid0 + g): sharding games over launches or
    GPUs does not change any game.  ``out`` may be a previous Playout of the same shape to reuse.
    ``totals``: optional int64 [4] device tensor, += (plies, sum of n_black - n_white, Black wins, White
    wins) over the games of this launch -- what play_a_game / store_batch_stats report
    (game_runner.py:194-199, learn_base.py:70-88).
    ``depth`` / ``depth_white``: search depths (1..SEARCH_MAX_DEPTH) of a POLICY_SEARCH side, Black's and White's;
    White's defaults to ``depth``.  A search side plays the move ``search`` returns, except on random plies,
    substituted plies and forced moves, which follow the greedy engine's rules.
    """
    searching = [p == POLICY_SEARCH for p in (policy, policy if policy_white is None else policy_white)]
    depth_w = depth if depth_white is None else depth_white
    for searches, d, side in zip(searching, (depth, depth_w), ("Black", "White")):
        if searches and not (d is not None and 1 <= int(d) <= SEARCH_MAX_DEPTH):
            raise ValueError("%s searches: its depth must be in 1..%d, got %r" % (side, SEARCH_MAX_DEPTH, d))
    if device is None:
        device = black0.device if black0 is not None else torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    n = int(n_games)
    if out is None:
        tb = torch.empty((t_max + 1, n), dtype=torch.int64, device=device) if trajectory else None
        tw = torch.empty((t_max + 1, n), dtype=torch.int64, device=device) if trajectory else None
        tm = torch.empty((t_max, n), dtype=torch.uint8, device=device) if trajectory else None
        out = Playout(n, t_max, tb, tw, tm, torch.empty(n, dtype=torch.int32, device=device),
                      torch.empty(n, dtype=torch.int64, device=device), torch.empty(n, dtype=torch.int64, device=device))
    a = _lib.PlayoutArgs()
    a.seed, a.gid0, a.n_games = seed & 0xFFFFFFFFFFFFFFFF, gid0 & 0xFFFFFFFFFFFFFFFF, n
    a.black0 = _opt(black0, torch.int64, n, "black0")
    a.white0 = _opt(white0, torch.int64, n, "white0")
    a.turn0 = _opt(turn0, torch.uint8, n, "turn0")
    a.policy, a.random_plies, a.n_rand_black, a.n_rand_white = policy, random_plies, n_rand_black, n_rand_white
    a.weights = _opt(weights, torch.float32, 40, "weights")
    a.policy_white = -1 if policy_white is None else policy_white      # White's engine (None = same as Black's)
    a.weights_white = _opt(weights_white, torch.float32, 40, "weights_white")
    a.t_max, a.stride = out.t_max, n
    a.traj_black = _opt(out.black, torch.int64, (out.t_max + 1) * n, "traj_black")
    a.traj_white = _opt(out.white, torch.int64, (out.t_max + 1) * n, "traj_white")
    a.traj_move = _opt(out.move, torch.uint8, out.t_max * n, "traj_move") if out.t_max > 0 else None
    a.nplies = _req(out.nplies, torch.int32, n, "nplies")
    a.final_black = _req(out.final_black, torch.int64, n, "final_black")
    a.final_white = _req(out.final_white, torch.int64, n, "final_white")
    a.totals = _opt(totals, torch.int64, 4, "totals")
    a.games_per_warp = games_per_warp                          # greedy engine: 0 = chosen from n_games
    a.summary = _opt(summary, torch.int16, n, "summary")        # per game: plies | (n_black - n_white) << 8
    with torch.cuda.device(device):
        stream = _stream(out.nplies)
        if any(searching):
            a.policy_white = policy if policy_white is None else policy_white   # (so White's depth is depth_w)
            a.search_depth = int(depth) if searching[0] else 0
            a.search_depth_white = int(depth_w) if searching[1] else 0
            ws, nbytes = _search_workspace(device, stream)      # the work counter: shared with ``search`` on this stream
            a.workspace, a.workspace_bytes = ctypes.c_void_p(ws.data_ptr()), nbytes
        _lib.check(_lib.lib().othello_playout(ctypes.byref(a), stream), "othello_playout")
    return out


_perft_ws = {}


def _perft_workspace(depth, device):
    nbytes = int(_lib.lib().othello_perft_workspace_bytes(depth))
    ws = _perft_ws.get(device)
    if ws is None or ws.numel() < nbytes:
        ws = _perft_ws[device] = torch.empty(nbytes, dtype=torch.uint8, device=device)
    return ws, nbytes


def perft(depth, black=START_BLACK, white=START_WHITE, turn=BLACK, device=None):
    """Node count of the legal-move tree to ``depth`` (pass = ply, game-over node = leaf)."""
    device = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
    ws, nbytes = _perft_workspace(depth, device)
    res = ctypes.c_uint64(0)
    with torch.cuda.device(device):
        _lib.check(_lib.lib().othello_perft(unsigned64(black), unsigned64(white), turn, depth, ctypes.c_void_p(ws.data_ptr()),
                                            nbytes, ctypes.byref(res), _stream(ws)), "othello_perft")
    return int(res.value)


def perft_part(depth, part, nparts, black=START_BLACK, white=START_WHITE, turn=BLACK, device=None):
    """This part's share of perft(depth), left ON the device: int64 [2] = (nodes, workspace-overflow flag).
    Only enqueues (othello_perft_async); the nparts shares add up to the node count."""
    device = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
    out = torch.zeros(2, dtype=torch.int64, device=device)
    if depth == 0:
        out[0] = 1 if part == 0 else 0
        return out
    ws, nbytes = _perft_workspace(depth, device)
    with torch.cuda.device(device):
        _lib.check(_lib.lib().othello_perft_async(unsigned64(black), unsigned64(white), turn, depth, part, nparts,
                                                  ctypes.c_void_p(ws.data_ptr()), nbytes, ctypes.c_void_p(out.data_ptr()),
                                                  _stream(ws)), "othello_perft_async")
    return out


def perft_distributed(depth, black=START_BLACK, white=START_WHITE, turn=BLACK, device=None):
    """perft with the depth-first stage split over the ranks of the default process group: every rank
    expands the (small) frontier itself, counts every world-th node, one all-reduce of a u64 (SURVEY 8e)."""
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    out = perft_part(depth, rank, world, black, white, turn, device)
    if world > 1:
        dist.all_reduce(out, op=dist.ReduceOp.SUM)
    nodes, overflow = (int(v) for v in out.cpu().tolist())
    if overflow:
        raise _lib.OthelloError(-2, "othello_perft_async")
    return nodes


NO_MOVE = 255                                    # OTHELLO_NO_MOVE: the game is over (or the position was refused)
SOLVE_MAX_EMPTIES = 24                           # OTHELLO_SOLVE_MAX_EMPTIES
SOLVE_REFUSED = -128                             # OTHELLO_SOLVE_REFUSED
_solve_ws = {}                                   # (device, stream) -> workspace: the work counter of one call at a time


def _solve_workspace(dev, stream):
    """the workspace of ``solve`` and ``solve_moves`` on (dev, stream): calls on one stream run one after the other, so
    they can share its counter; calls on different streams may overlap, so each stream has its own"""
    nbytes = int(_lib.lib().othello_solve_workspace_bytes())
    ws = _solve_ws.get((dev, stream.value))
    if ws is None:
        ws = _solve_ws[(dev, stream.value)] = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    return ws, nbytes


def solve(black, white, turn=None, nodes=False):
    """Exact endgame values (othello_solve): (value int32 [n], move uint8 [n], nodes int64 [n] or None).

    value = own - opponent discs at the end of perfect play, own = the side to move (``turn``: uint8 [n], 1 = Black,
    None = Black to move everywhere); empty squares left at the end are not given to the winner.  move = the lowest
    square reaching the value, PASS when the mover must pass, NO_MOVE when the game is over.  Positions with more
    than SOLVE_MAX_EMPTIES empties or overlapping colours get SOLVE_REFUSED / NO_MOVE.  ``nodes``: also return the
    positions the search visited, per position (benchmarking)."""
    n = black.numel()
    dev = black.device
    value = torch.empty(n, dtype=torch.int32, device=dev)
    move = torch.empty(n, dtype=torch.uint8, device=dev)
    cnt = torch.empty(n, dtype=torch.int64, device=dev) if nodes else None
    with torch.cuda.device(dev):
        stream = _stream(black)
        ws, nbytes = _solve_workspace(dev, stream)
        _lib.check(_lib.lib().othello_solve(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"), _opt(turn, torch.uint8, n, "turn"),
            _req(value, torch.int32, n, "value"), _req(move, torch.uint8, n, "move"), _opt(cnt, torch.int64, n, "nodes"),
            n, _req(ws, torch.uint8, nbytes, "workspace"), nbytes, stream), "othello_solve")
    return value, move, cnt


SEARCH_MAX_DEPTH = 12                            # OTHELLO_SEARCH_MAX_DEPTH
_search_ws = {}                                  # (device, stream) -> workspace: the work counter of one call at a time


def _search_workspace(dev, stream):
    """the workspace of ``search``, ``search_moves`` and of search playouts on (dev, stream): calls on one stream run one after the
    other, so they can share its counter; calls on different streams may overlap, so each stream has its own"""
    nbytes = int(_lib.lib().othello_search_workspace_bytes())
    ws = _search_ws.get((dev, stream.value))
    if ws is None:
        ws = _search_ws[(dev, stream.value)] = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    return ws, nbytes


def search(black, white, weights, depth, turn=None, nodes=False):
    """Depth-limited midgame search on the linear evaluation (othello_search): (value float32 [n], move uint8 [n],
    nodes int64 [n] or None).

    Every node is scored with ``weights`` (float32 [4][10] on the device) from the side to move at the root (``turn``:
    uint8 [n], 1 = Black, None = Black to move everywhere); a pass is a ply and uses one level of ``depth``
    (1..SEARCH_MAX_DEPTH).  value = the minimax value, move = the lowest square reaching it, PASS when the mover must
    pass, NO_MOVE when the game is over.  depth 1 is the greedy policy.  Positions with overlapping colours get NaN /
    NO_MOVE.  ``nodes``: also return the positions the search visited, per position (benchmarking)."""
    if not 1 <= int(depth) <= SEARCH_MAX_DEPTH:
        raise ValueError("depth must be in 1..%d, got %r" % (SEARCH_MAX_DEPTH, depth))
    n = black.numel()
    dev = black.device
    value = torch.empty(n, dtype=torch.float32, device=dev)
    move = torch.empty(n, dtype=torch.uint8, device=dev)
    cnt = torch.empty(n, dtype=torch.int64, device=dev) if nodes else None
    with torch.cuda.device(dev):
        stream = _stream(black)
        ws, nbytes = _search_workspace(dev, stream)
        _lib.check(_lib.lib().othello_search(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"), _opt(turn, torch.uint8, n, "turn"),
            _req(weights, torch.float32, 40, "weights"), int(depth), _req(value, torch.float32, n, "value"),
            _req(move, torch.uint8, n, "move"), _opt(cnt, torch.int64, n, "nodes"), n,
            _req(ws, torch.uint8, nbytes, "workspace"), nbytes, stream), "othello_search")
    return value, move, cnt


MOVE_SLOTS = 65                                  # OTHELLO_MOVE_SLOTS: a row per position, squares 0..63 and PASS


def search_moves(black, white, weights, depth, turn=None, nodes=False):
    """The search value of every move (othello_search_moves): (values float32 [n][MOVE_SLOTS], nodes int64
    [n][MOVE_SLOTS] or None).

    values[i][s] = the minimax value of the subtree after square s, searched to ``depth`` - 1 further plies with every
    node scored from the root mover's side, as ``search`` scores it; values[i][PASS] = the passed position's value when
    the mover must pass; NaN where there is no such move (and in every entry of a game-over position or of overlapping
    colours).  The row's maximum and lowest arg-max are ``search``'s value and move.  Only enqueues."""
    if not 1 <= int(depth) <= SEARCH_MAX_DEPTH:
        raise ValueError("depth must be in 1..%d, got %r" % (SEARCH_MAX_DEPTH, depth))
    n = black.numel()
    dev = black.device
    values = torch.empty((n, MOVE_SLOTS), dtype=torch.float32, device=dev)
    cnt = torch.empty((n, MOVE_SLOTS), dtype=torch.int64, device=dev) if nodes else None
    with torch.cuda.device(dev):
        stream = _stream(black)
        ws, nbytes = _search_workspace(dev, stream)
        _lib.check(_lib.lib().othello_search_moves(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"), _opt(turn, torch.uint8, n, "turn"),
            _req(weights, torch.float32, 40, "weights"), int(depth), _req(values, torch.float32, MOVE_SLOTS * n, "values"),
            _opt(cnt, torch.int64, MOVE_SLOTS * n, "nodes"), n, _req(ws, torch.uint8, nbytes, "workspace"), nbytes,
            stream), "othello_search_moves")
    return values, cnt


def solve_moves(black, white, turn=None, nodes=False):
    """The perfect-play value of every move (othello_solve_moves): (values int32 [n][MOVE_SLOTS], nodes int64
    [n][MOVE_SLOTS] or None).

    values[i][s] = the value after square s from the mover's side (minus ``solve`` of the child); values[i][PASS] =
    ``solve``'s value when the mover must pass; SOLVE_REFUSED where there is no such move, and in every entry of a
    position with more than SOLVE_MAX_EMPTIES empties, a game-over position or overlapping colours.  The row's maximum
    and lowest arg-max are ``solve``'s value and move.  Only enqueues."""
    n = black.numel()
    dev = black.device
    values = torch.empty((n, MOVE_SLOTS), dtype=torch.int32, device=dev)
    cnt = torch.empty((n, MOVE_SLOTS), dtype=torch.int64, device=dev) if nodes else None
    with torch.cuda.device(dev):
        stream = _stream(black)
        ws, nbytes = _solve_workspace(dev, stream)
        _lib.check(_lib.lib().othello_solve_moves(
            _req(black, torch.int64, n, "black"), _req(white, torch.int64, n, "white"), _opt(turn, torch.uint8, n, "turn"),
            _req(values, torch.int32, MOVE_SLOTS * n, "values"), _opt(cnt, torch.int64, MOVE_SLOTS * n, "nodes"), n,
            _req(ws, torch.uint8, nbytes, "workspace"), nbytes, stream), "othello_solve_moves")
    return values, cnt


def decay_table(t_max, lam=0.90):
    """decay[k] = lam ** k in fp64, evaluated by CPython exactly like `self.l ** turn_left`
    (progress_position_moves_learn.py:24,55)."""
    return np.array([lam ** k for k in range(t_max + 1)], dtype=np.float64)


N_ACC = 80                                       # OTHELLO_ACC: exact integer accumulators per phase shard
_decay_cache = {}


def decay_tensor(t_max, lam, device):
    """decay_table on the device, uploaded once per (t_max, lam, device)"""
    key = (int(t_max), float(lam), str(device))
    t = _decay_cache.get(key)
    if t is None:
        t = _decay_cache[key] = torch.from_numpy(decay_table(t_max, lam)).to(device)
    return t


def learn_accumulate(po, acc=None, lam=0.90):
    """Exact per-shard normal-equation accumulators int64 [4][80] (+=) of a Playout's trajectories
    (include/othello_b200.h: othello_learn_accumulate).  Integer sums: additive over any split of the
    games, bit for bit; ``learn_stats`` turns them into the doubles the solvers read."""
    dev = po.nplies.device
    if po.black is None:
        raise ValueError("learn_accumulate needs a Playout with trajectories")
    if acc is None:
        acc = torch.zeros((4, N_ACC), dtype=torch.int64, device=dev)
    decay = decay_tensor(po.t_max, lam, dev)
    n = po.n_games
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().othello_learn_accumulate(
            _req(po.black, torch.int64, (po.t_max + 1) * n, "traj_black"),
            _req(po.white, torch.int64, (po.t_max + 1) * n, "traj_white"),
            _req(po.nplies, torch.int32, n, "nplies"), _req(po.final_black, torch.int64, n, "final_black"),
            _req(po.final_white, torch.int64, n, "final_white"), n, n, po.t_max,
            _req(decay, torch.float64, po.t_max + 1, "decay"), _req(acc, torch.int64, 4 * N_ACC, "acc"),
            _stream(acc)), "othello_learn_accumulate")
    return acc


def learn_stats(acc, out=None):
    """accumulators int64 [4][80] -> statistics float64 [4][112] (XtX[10][10], Xty[10], n, sum y^2)"""
    out = torch.empty((4, 112), dtype=torch.float64, device=acc.device) if out is None else out
    with torch.cuda.device(acc.device):
        _lib.check(_lib.lib().othello_learn_stats(_req(acc, torch.int64, 4 * N_ACC, "acc"),
                                                  _req(out, torch.float64, 448, "stats"), _stream(acc)),
                   "othello_learn_stats")
    return out


def learn_solve(stats, prev_weights, weights_out=None):
    """The four per-phase fits on the device (no host round trip): returns (weights float32 [4][10],
    params int32 [36], fits float64 [4][16] = coef[9], intercept, rmse, r2, n, 0, 0, 0)."""
    dev = stats.device
    weights_out = torch.empty((4, 10), dtype=torch.float32, device=dev) if weights_out is None else weights_out
    params = torch.empty(36, dtype=torch.int32, device=dev)
    fits = torch.empty((4, 16), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().othello_learn_solve(
            _req(stats, torch.float64, 448, "stats"), _req(prev_weights, torch.float32, 40, "prev_weights"),
            _req(weights_out, torch.float32, 40, "weights_out"), _req(params, torch.int32, 36, "params"),
            _req(fits, torch.float64, 64, "fits"), _stream(stats)), "othello_learn_solve")
    return weights_out, params, fits


def learn_refit(acc, prev_weights, weights_out=None, clear=True, stats_out=None, params=None, fits=None):
    """accumulators int64 [4][80] -> (weights, params, fits) in one launch (othello_learn_refit); ``clear`` zeroes
    the accumulators for the next iteration, ``stats_out`` (float64 [4][112]) also receives the statistics."""
    dev = acc.device
    weights_out = torch.empty((4, 10), dtype=torch.float32, device=dev) if weights_out is None else weights_out
    params = torch.empty(36, dtype=torch.int32, device=dev) if params is None else params
    fits = torch.empty((4, 16), dtype=torch.float64, device=dev) if fits is None else fits
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().othello_learn_refit(
            _req(acc, torch.int64, 4 * N_ACC, "acc"), 1 if clear else 0, _opt(stats_out, torch.float64, 448, "stats_out"),
            _req(prev_weights, torch.float32, 40, "prev_weights"), _req(weights_out, torch.float32, 40, "weights_out"),
            _req(params, torch.int32, 36, "params"), _req(fits, torch.float64, 64, "fits"), _stream(acc)),
            "othello_learn_refit")
    return weights_out, params, fits


def int32_peak(device=None, iters=4096, blocks_per_sm=8, threads=256, repeats=5, dual=False):
    """Measured INT32 throughput (lane-ops/s) of this GPU: the integer roofline denominator.

    dual=False: ALU pipe only (LOP3/SHF); dual=True: ALU + FMA pipes (LOP3 + IMAD, 1:1).  One round
    of either micro-benchmark kernel (csrc/peak.cu) is 32 integer lane-ops per thread.
    """
    device = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    blocks = sms * blocks_per_sm
    sink = torch.empty(blocks * threads, dtype=torch.int32, device=device)
    L = _lib.lib()
    kern = L.othello_int32_dual_peak_kernel if dual else L.othello_int32_peak_kernel
    best = None
    with torch.cuda.device(device):
        st = _stream(sink)
        for _ in range(2):
            _lib.check(kern(ctypes.c_void_p(sink.data_ptr()), blocks, threads, iters, st), "peak")
        for _ in range(repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(kern(ctypes.c_void_p(sink.data_ptr()), blocks, threads, iters, st), "peak")
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
    ops = 32.0 * iters * blocks * threads
    return ops / (best * 1e-3)
