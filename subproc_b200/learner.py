"""The data-parallel learner: per-phase linear regression from statistics accumulated on the GPUs.

Replaces, for BASELINE config 5, the reference's learning round trip
(progress_position_moves_learn.py): every position of every self-play game contributes its
``counts()`` features and its discounted final score (``__update_state_for_a_book`` :37-48,
``l = 0.90`` :24) to the normal equations of its disc-count shard (:112-113); where the reference
enqueues four pyres jobs and polls Redis for their answers (:115-158), the ranks here exchange ONE
all-reduce of 4 x 112 doubles and every rank solves the four 10 x 10 systems itself.

What is kept from the reference, to the letter:
  * the regressors (mobility, a..h) + intercept -- ``LinearRegression(fit_intercept=True)`` (:167);
    rank-deficient shards (square classes nobody occupies yet) get sklearn's minimum-norm solution;
  * ``param = coef * 127 / max|coef|`` with the intercept dropped (:180-181);
  * ``int(x)`` truncation toward zero when the parameters are stored (:196-203), the field order
    'A'.. and the ``(header, w0..w35)`` tuple of ``read_parameters`` (:211-224).
What differs, and why: the reference fits on <= 50 000 keys drawn from its smoothed value table with
Python's ``random`` and ``sklearn.utils.resample`` (:66-86,160-165) -- unpinned RNG, no test in the
reference fixes any output -- so this path regresses on the full sample stream instead (every
position once per side).  The order-dependent table itself is ``subproc_b200.value_table``.
"""
import math

import numpy as np

from . import parameter as parameter_mod

PHASE_SHARDS = [(0, 16), (17, 32), (33, 48), (49, 64)]        # progress_position_moves_learn.py:112-113
N_X = 10                                                        # mobility, a..h, intercept
N_STATS = 112                                                   # XtX[10][10], Xty[10], n, sum y^2


def unpack_stats(row):
    row = np.asarray(row, dtype=np.float64)
    return row[:100].reshape(10, 10), row[100:110], float(row[110]), float(row[111])


def solve_shard(row, rcond=1e-12):
    """OLS with intercept from one shard's statistics; minimum-norm when the Gram matrix is singular
    (what sklearn's lstsq-based LinearRegression returns).  -> dict(coef[9], intercept, rmse, r2, n)"""
    xtx, xty, n, syy = unpack_stats(row)
    if n <= 0:
        return dict(coef=np.zeros(9), intercept=0.0, rmse=float('nan'), r2=float('nan'), n=0)
    xbar = xtx[:9, 9] / n                                       # column of ones: sum x_i
    ybar = xty[9] / n
    sxx = xtx[:9, :9] - n * np.outer(xbar, xbar)                # centred Gram matrix
    sxy = xty[:9] - n * xbar * ybar
    coef = np.zeros(9)
    live = np.flatnonzero(np.diag(sxx) > 0)                     # constant columns (e.g. classes nobody owns yet) get 0
    if live.size:
        sub = sxx[np.ix_(live, live)]
        lam, q = np.linalg.eigh((sub + sub.T) * 0.5)
        keep = lam > rcond * max(lam.max(), 0.0)
        inv = np.zeros_like(lam)
        inv[keep] = 1.0 / lam[keep]
        coef[live] = q @ (inv * (q.T @ sxy[live]))
    intercept = ybar - float(xbar @ coef)
    w = np.concatenate([coef, [intercept]])
    sse = max(syy - 2.0 * float(w @ xty) + float(w @ xtx @ w), 0.0)
    sst = syy - n * ybar * ybar
    return dict(coef=coef, intercept=intercept, rmse=math.sqrt(sse / n),
                r2=(1.0 - sse / sst) if sst > 0 else float('nan'), n=int(n))


def fit_from_stats(stats):
    """stats [4][112] (numpy or tensor) -> list of 4 shard fits."""
    if hasattr(stats, "detach"):
        stats = stats.detach().cpu().numpy()
    return [solve_shard(stats[s]) for s in range(4)]


def scale_param(coef):
    """coef * 127 / max|coef| (progress_position_moves_learn.py:180-181)"""
    m = float(np.max(np.abs(coef)))
    if m == 0.0:
        return tuple(0.0 for _ in coef)
    k = 127 / m
    return tuple(float(c) * k for c in coef)


def stored_parameters(params_rows):
    """__store_parameters: flatten the 4 rows, int() truncation toward zero (:196-203)"""
    return [int(x) for row in params_rows for x in row]


N_ACC = 80                                                      # OTHELLO_ACC (include/othello_b200.h)
_KX = 10
_FP_BASE = 56


def _pair(i, j):
    return i * _KX - i * (i - 1) // 2 + (j - i)


def stats_from_acc(acc):
    """othello_learn_stats on the host: exact integer accumulators [4][80] (numpy / CPU tensor) -> the
    [4][112] doubles (XtX[10][10], Xty[10], n, sum y^2), each the correctly rounded image of its integer
    sum (Python integers: no intermediate rounding)."""
    if hasattr(acc, "detach"):
        acc = acc.detach().cpu().numpy()
    acc = np.asarray(acc, dtype=np.int64).reshape(4, N_ACC)
    out = np.zeros((4, N_STATS), dtype=np.float64)
    for s in range(4):
        a = [int(v) for v in acc[s]]
        for i in range(_KX):
            for j in range(_KX):
                out[s, i * _KX + j] = float(a[_pair(min(i, j), max(i, j))])
        out[s, 110] = float(a[_pair(9, 9)])
        for k in range(10):                                     # Xty[0..8], then sum y^2
            total = (a[_FP_BASE + 2 * k] << 32) + a[_FP_BASE + 2 * k + 1]
            out[s, 111 if k == 9 else 100 + k] = total / float(1 << 40)      # int / float: one rounding
    return out


def allreduce_stats(stats):
    """sum the per-rank statistics / accumulators over all ranks (NCCL for CUDA tensors, gloo for CPU
    tensors).  A no-op in a single process.  On the int64 accumulators the sum is exact, so every rank
    count gives the same bits; on doubles it is the usual tolerance-level reduction."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def shard_of_games(total_games, rank, world):
    """contiguous split of global game ids: rank r plays [lo, hi) -- g // (B / ngpu) of SURVEY 8(e)"""
    per = (total_games + world - 1) // world
    lo = min(rank * per, total_games)
    return lo, min(lo + per, total_games)


def batch_stats(black_discs, white_discs, black_name='black', white_name='white', params_used=''):
    """The payload of LearnBasePlus.store_batch_stats (learn_base.py:58-110) from the final disc counts
    of a batch of games, in book order.

    Kept to the letter, including the reference's white-win test ``white_discs > black_wins``
    (learn_base.py:77 compares White's discs with the running COUNT of Black wins); the count a reader
    would expect is returned under 'white_wins_by_discs'."""
    b = np.asarray(black_discs, dtype=np.int64)
    w = np.asarray(white_discs, dtype=np.int64)
    n = len(b)
    black_won = b > w
    wins_before = np.cumsum(black_won) - black_won           # black_wins when the elif is evaluated
    white_won_ref = (~black_won) & (w > wins_before)
    diff = (b - w).tolist()
    return {
        black_name + '_win_rate': float(black_won.sum()) / float(n),
        white_name + '_win_rate': float(white_won_ref.sum()) / float(n),
        'min_disc_diff': min(diff), 'max_disc_diff': max(diff),
        'avg_disc_diff': float(sum(diff)) / float(n),
        'params_used': params_used, 'diffs': sorted(diff),
        'white_wins_by_discs': int((w > b).sum()),
    }


def _self_play_policy(depth):
    """the engine of self-play: greedy, or the midgame search when a depth is given"""
    from . import ops
    return ops.POLICY_GREEDY if depth is None else ops.POLICY_SEARCH


class ProgressPositionMovesLearn(object):
    """The reference learner's public surface (name / configure / fit_parameter / read_parameters,
    learn_base.py:8-33, progress_position_moves_learn.py:19-35) over on-GPU self-play."""

    def __init__(self):
        self.conf = {}
        self.a = 0.03
        self.b = 0.003
        self.l = 0.90
        self.parameter = parameter_mod.ProgressPositionMovesParameter()
        self.params = None                      # stored ints, flat list of 36
        self.last_fits = None
        self.last_stats = None
        self.last_processed_id = -1

    def name(self):
        return 'progresspositionmovelearn'

    def configure(self, conf_dict):
        self.conf = conf_dict
        self.parameter.configure(conf_dict)

    def last_processed(self):
        return self.last_processed_id

    def read_parameters(self):
        """(header, w0..w35) (:211-224); the default rows until something has been learnt"""
        if self.params is None:
            self.params = stored_parameters(self.parameter.default_value())
        return tuple([self.parameter.header()] + list(self.params))

    def weights_table(self):
        return self.parameter.weights_table(self.read_parameters())

    def store_batch_stats(self, playout, black_name='b200', white_name='b200', params_used='No Hamlet'):
        """win rates / disc differences of a batch (learn_base.py:58-110), counts from the GPU"""
        c = playout.final_counts().cpu().numpy()
        self.last_batch_stats = batch_stats(c[:, 0], c[:, 1], black_name, white_name, params_used)
        return self.last_batch_stats

    # ---- one learning iteration ------------------------------------------------------------
    def accumulate(self, playout, acc=None):
        """exact integer accumulators int64 [4][80] of a playout's trajectories (+= into ``acc``)"""
        from . import ops
        return ops.learn_accumulate(playout, acc=acc, lam=self.l)

    def learn_from_acc(self, acc, book_id=None):
        """all-reduce of the exact accumulators (320 int64 -- the ranks' only exchange, replacing the Redis
        `fitting:*` polling of progress_position_moves_learn.py:131-150) -> statistics -> refit.  Integer
        sums: the learnt parameters are identical for every rank count."""
        acc = allreduce_stats(acc)
        if getattr(acc, "is_cuda", False):
            from . import ops
            stats = ops.learn_stats(acc)
        else:
            stats = stats_from_acc(acc)
        return self._refit(stats, book_id)

    def fit_parameter(self, phase_from, phase_to):
        """(mse, score, param, nsample) of one shard, like the reference's worker job (:160-184),
        from the statistics of the last iteration."""
        s = PHASE_SHARDS.index((phase_from, phase_to))
        fit = self.last_fits[s]
        return fit['rmse'], fit['r2'], scale_param(fit['coef']), fit['n']

    def learn_from_stats(self, stats, book_id=None):
        """all-reduce of fp64 statistics [4][112] -> 4 solves -> scale to +-127 -> int() -> stored
        parameters (for statistics that do not come from the accumulators, e.g. samples of the value table)"""
        return self._refit(allreduce_stats(stats), book_id)

    def _refit(self, stats, book_id=None):
        self.last_stats = stats
        self.last_fits = fit_from_stats(stats)
        rows = []
        old = np.asarray(self.read_parameters()[1:], dtype=np.float64).reshape(4, 9)
        for s, (lo, hi) in enumerate(PHASE_SHARDS):
            if self.last_fits[s]['n'] > 0:
                rows.append(self.fit_parameter(lo, hi)[2])
            else:
                rows.append(tuple(old[s]))
        self.params = stored_parameters(rows)
        if book_id is not None:
            self.last_processed_id = book_id
        return rows

    def self_play_iterations_on_device(self, n_iterations, games_per_rank, seed=0, first_iteration=0, random_plies=10,
                                       device=None, rank=0, world=1, t_max=120, depth=None):
        """config 5 without host round trips: every iteration is playout -> statistics -> all-reduce ->
        othello_learn_refit -> the next playout reads the new table straight from device memory.  The
        host only enqueues; parameters are copied back once at the end.  Same arithmetic as
        ``self_play_iteration`` on identical statistics (the integer parameters may differ by one where a
        scaled coefficient sits on an integer boundary: two eigen-solvers, last-ulp differences).
        ``depth``: None plays greedy games; 1..12 plays search self-play at that depth on the current table (the
        whole game on the device, so the loop still never waits for the host)."""
        import torch
        from . import ops
        dev = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
        w = torch.from_numpy(self.weights_table()).to(dev)
        acc = torch.zeros((4, N_ACC), dtype=torch.int64, device=dev)
        stats = torch.empty((4, 112), dtype=torch.float64, device=dev)
        po = params = fits = None
        for it in range(first_iteration, first_iteration + n_iterations):
            gid0 = (it * world + rank) * games_per_rank
            po = ops.playout(games_per_rank, seed=seed, gid0=gid0, device=dev, policy=_self_play_policy(depth),
                             random_plies=random_plies, weights=w, t_max=t_max, out=po, depth=depth)
            ops.learn_accumulate(po, acc=acc, lam=self.l)
            allreduce_stats(acc)
            # statistics + four regressions + clearing the accumulators: one launch, weights updated in place
            w, params, fits = ops.learn_refit(acc, w, weights_out=w, clear=True, stats_out=stats, params=params, fits=fits)
        self.params = [int(v) for v in params.cpu().tolist()]
        f = fits.cpu().numpy()
        self.last_fits = [dict(coef=f[s, :9].copy(), intercept=float(f[s, 9]), rmse=float(f[s, 10]), r2=float(f[s, 11]),
                               n=int(f[s, 12])) for s in range(4)]
        self.last_stats = stats
        # the id of the last game of the last iteration over ALL ranks, so every rank's checkpoint agrees
        self.last_processed_id = (first_iteration + n_iterations) * world * games_per_rank - 1
        return po

    # ---- checkpoint / resume ------------------------------------------------------------------
    def save(self, path):
        """Everything the reference keeps in Redis for this learner (progress_position_moves_learn.py:
        188-224 and the value table :52): last processed book id, the stored parameters, the table."""
        import torch
        table = getattr(self, 'table', None)
        torch.save({'name': self.name(), 'last_processed': self.last_processed_id, 'params': self.params,
                    'a': self.a, 'l': self.l,
                    'table_keys': None if table is None else table.keys.cpu(),
                    'table_values': None if table is None else table.values.cpu()}, path)

    def load(self, path, device=None):
        import torch
        from . import value_table
        state = torch.load(path, map_location='cpu')
        if state['name'] != self.name():
            raise ValueError("checkpoint belongs to learner %r" % state['name'])
        self.last_processed_id, self.params, self.a, self.l = state['last_processed'], state['params'], state['a'], state['l']
        self.table = None
        if state['table_keys'] is not None:
            self.table = value_table.ValueTable(device=device, a=self.a, lam=self.l)
            self.table.load_state(state['table_keys'], state['table_values'])
        return self

    # ---- the reference's book-driven entry point ---------------------------------------------
    def learn_and_update_batch(self, books, device=None, sample=50000, seed=0):
        """LearnBasePlus.learn_and_update_batch (progress_position_moves_learn.py:88-101) on the
        reference's own input: ``books`` = [(book_id, records, meta)] with ``records`` as learn_books
        hands them over -- sorted by turn and REVERSED, records[0] the terminal position
        (replearn.py:37-38).  Every (record, side) updates the value table in the reference's order
        (:37-48), then the four shards are refitted on samples of the table (:115-158 -> value_table.
        fit_parameter) and stored with int() truncation (:196-209).  Returns (mses, scores, params,
        nsamples) like __fit_parameters."""
        import torch
        from . import books as books_mod
        from . import ops, value_table
        dev = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
        if getattr(self, 'table', None) is None:
            self.table = value_table.ValueTable(device=dev, a=self.a, lam=self.l)
        flat, targets = [], []
        last_book_id = -1
        for book_id, records, _meta in books:
            last_turn = int(records[0]['turn'])
            flat.extend(records)
            targets.append((len(records), last_turn, [int(r['turn']) for r in records]))
            last_book_id = book_id
        if flat:
            black, white, _who, _turns = books_mod.positions_from_books(flat, device=dev)
            n = black.numel()
            side_o = torch.full((n,), ops.BLACK, dtype=torch.uint8, device=dev)
            fo = ops.features(black, white, side_o).cpu().numpy()
            fx = ops.features(black, white, side_o + 1).cpu().numpy()
            keys = np.empty(2 * n, dtype=np.int64)
            vals = np.empty(2 * n, dtype=np.float64)
            at = 0
            for count, last_turn, turns in targets:
                nb, nw = int(fo[at, 2:].sum()), int(fx[at, 2:].sum())          # records[0] is terminal: its disc counts
                for j in range(count):
                    left = last_turn - turns[j]
                    keys[2 * (at + j)] = value_table.pack_key(fo[at + j])
                    vals[2 * (at + j)] = float(nb - nw) * (self.l ** left)     # side 'O', value_for_black (:40-47)
                    keys[2 * (at + j) + 1] = value_table.pack_key(fx[at + j])
                    vals[2 * (at + j) + 1] = float(nw - nb) * (self.l ** left)
                at += count
            self.table.update(torch.from_numpy(keys).to(dev), torch.from_numpy(vals).to(dev))
        mses, scores, params, nsamples = [], [], [], []
        old = np.asarray(self.read_parameters()[1:], dtype=np.float64).reshape(4, 9)
        for s, (lo, hi) in enumerate(PHASE_SHARDS):
            mse, score, param, nsample = self.table.fit_parameter(lo, hi, num=sample, seed=seed + s)
            if nsample == 0:                                   # nothing seen in this phase yet: keep the stored row
                param = tuple(float(v) for v in old[s])
            mses.append(mse); scores.append(score); params.append(param); nsamples.append(nsample)
        self.params = stored_parameters(params)
        self.last_processed_id = last_book_id
        return mses, scores, params, nsamples

    def self_play_iteration_table(self, n_games, seed=0, iteration=0, random_plies=10, device=None, t_max=120,
                                  sample=50000):
        """One learning iteration with the REFERENCE's learning semantics (single GPU): greedy self-play with the
        current weights, every (position, side) smooths the order-dependent value table in the reference's order
        (progress_position_moves_learn.py:37-62,88-91), then each shard is refitted on a sample of <= 50 000
        distinct table entries (:66-86,160-184) and stored with int() truncation (:196-209).
        Returns (playout, (mses, scores, params, nsamples))."""
        import torch
        from . import ops, value_table
        dev = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
        if getattr(self, 'table', None) is None:
            self.table = value_table.ValueTable(device=dev, a=self.a, lam=self.l)
        w = torch.from_numpy(self.weights_table()).to(dev)
        gid0 = iteration * n_games
        po = ops.playout(n_games, seed=seed, gid0=gid0, device=dev, policy=ops.POLICY_GREEDY,
                         random_plies=random_plies, weights=w, t_max=t_max)
        self.table.update_from_playout(po)
        old = np.asarray(self.read_parameters()[1:], dtype=np.float64).reshape(4, 9)
        mses, scores, params, nsamples = [], [], [], []
        for s, (lo, hi) in enumerate(PHASE_SHARDS):
            mse, score, param, nsample = self.table.fit_parameter(lo, hi, num=sample, seed=seed + 4 * iteration + s)
            if nsample == 0:
                param = tuple(float(v) for v in old[s])
            mses.append(mse); scores.append(score); params.append(param); nsamples.append(nsample)
        self.params = stored_parameters(params)
        self.last_processed_id = gid0 + n_games - 1
        return po, (mses, scores, params, nsamples)

    def self_play_iteration(self, games_per_rank, seed=0, iteration=0, random_plies=10, device=None, rank=0,
                            world=1, t_max=120, depth=None):
        """config 5: greedy self-play with the current weights on this rank's shard of game ids,
        statistics, all-reduce, refit.  Returns (playout, new parameter rows).  ``depth`` (1..12): search
        self-play at that depth instead, with the same random plies and game ids (depth 1 plays the greedy games)."""
        import torch
        from . import ops
        dev = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
        w = torch.from_numpy(self.weights_table()).to(dev)
        gid0 = (iteration * world + rank) * games_per_rank
        po = ops.playout(games_per_rank, seed=seed, gid0=gid0, device=dev, policy=_self_play_policy(depth),
                         random_plies=random_plies, weights=w, t_max=t_max, depth=depth)
        acc = self.accumulate(po)
        rows = self.learn_from_acc(acc, book_id=(iteration + 1) * world * games_per_rank - 1)
        return po, rows
