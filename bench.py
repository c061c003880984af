#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched Othello hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--games G] [--dump-outputs DIR]

Workload (config.workload = "config3_random_playout"): G = 2**20 lock-step random-playout games
PER GPU from the standard opening, every position and move written to HBM (SoA trajectory).  A
"step" is one launch of the playout kernel over one fresh batch of G games (new game ids every
step).  Games are independent, so N GPUs run N shards with no data-path collective ("weak").

    value   = positions/s = sum over ranks and steps of plies played / max-over-ranks device time
    e2e     = the same through the host-buffer C ABI (othello_playout_host): start positions come
              from pinned host memory, per-game results (plies, final position) go back to host
              memory, trajectories stay in HBM -- copies inside the timed region
    roofline= integer roofline of the playout kernel: frac = executed thread instructions per second
              (positions/s x the ncu-measured instructions per position, profiles/playout_kernel_costs.json)
              over the integer issue peak measured live by csrc/peak.cu (ALU + FMA pipes co-issuing
              LOP3 + IMAD); the canonical 512 INT32 lane-ops per position-step of SURVEY.md 8d are
              reported next to it as `algorithmic_*` (the kernel executes fewer), plus the HBM write-out
              rate (17 B per position) against MEASURED_PEAKS.json
    cpu_baseline = the reference's own board.py (oracle/_ref, py3 transcription) playing the same
              kind of games on all host cores for a bounded time (N=1, rank 0 only)

`--impl reference` times only that CPU path and prints the same JSON shape.

`--dump-outputs DIR` writes what the last timed launch returned (nplies, final positions and trajectories of a fixed
sample of its games, see sample_outputs) and the batch totals of all timed steps, from which `value` is computed, as
DIR/<name>.npy.  The games of a step depend only on --games, --warmup and
--steps, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "othello_positions_per_sec_legalgen_step"
UNIT = "positions/s"
LANE_OPS_PER_POSITION = 512          # SURVEY.md 8(d): 256 64-bit bit-ops per legal-gen + flip
BYTES_PER_POSITION = 17              # black u64 + white u64 + move u8 written per ply
T_MAX = 120


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference's board.py on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """plays seeded random games (bare loop: puttables -> choose -> put_s -> is_game_over) until the
    deadline; returns (plies, games).  Runs in a multiprocessing worker."""
    kind, seed, gid0, budget_s, max_games = args
    full_path = kind == "reference_full"
    t_end = time.perf_counter() + budget_s
    plies = games = 0
    if kind.startswith("reference"):
        from oracle import refshim, make_golden as mg
        rb = refshim.load().board
        while time.perf_counter() < t_end and games < max_games:
            B = rb.Board()
            key = mg.rng_key(seed, gid0 + games)
            t = 0
            while not B.is_game_over():
                moves = B.puttables(B.turn)
                if moves:
                    x, y = moves[mg.below(mg.rng_draw(key, t, 1), len(moves))]
                    B.put_s(B.handstr_from_coord(x, y))
                else:
                    B.put_s('ps')
                if full_path:
                    # what play_a_turn adds per ply (game_runner.py:154-163 + RedisRecorder.add,
                    # game_recorder.py:107-114): the printed board, the serialised record, its end flag
                    str(B)
                    {'book': B.serialize_board(), 'whosturn': B.serialize_turn(), 'turn': B.nturn,
                     'end': B.is_game_over()}
                t += 1
            plies += t
            games += 1
    else:
        from oracle import lib as orc
        while time.perf_counter() < t_end and games < max_games:
            r = orc.playout(seed, gid0 + games, 64, trajectory=False)
            plies += int(r['nplies'].sum())
            games += 64
    return plies, games


def play_a_game_through(board_module, seed, gid, mg):
    """one random-vs-random game driven like GameRunner.play_a_turn (game_runner.py:154-163) with a
    RedisRecorder-style record per ply (game_recorder.py:107-114), on ANY module with the reference's
    `Board` interface; returns (plies, final n_black, final n_white)"""
    B = board_module.Board()
    key = mg.rng_key(seed, gid)
    t = 0
    while not B.is_game_over():
        moves = B.puttables(B.turn)
        if moves:
            x, y = moves[mg.below(mg.rng_draw(key, t, 1), len(moves))]
            B.put_s(B.handstr_from_coord(x, y))
        else:
            B.put_s('ps')
        str(B)
        {'book': B.serialize_board(), 'whosturn': B.serialize_turn(), 'turn': B.nturn, 'end': B.is_game_over()}
        t += 1
    return t, B.n_black(), B.n_white()


def config1_facade(n_games=20):
    """BASELINE config 1: single games through the drop-in `subproc_b200.board.Board` (one kernel launch per
    change of position) next to the reference's own board.py on one host core, same seeded games."""
    from oracle import refshim, make_golden as mg
    from subproc_b200 import board as b200_board
    out = {"games": n_games, "driver": "puttables -> put_s -> str(board) -> serialize -> is_game_over per ply "
                                       "(game_runner.py:154-163, game_recorder.py:107-114)"}
    play_a_game_through(b200_board, 7, 999, mg)                     # context creation, first launches
    t0 = time.perf_counter()
    got = [play_a_game_through(b200_board, 7, g, mg) for g in range(n_games)]
    dt = time.perf_counter() - t0
    plies = sum(g[0] for g in got)
    out["b200_facade"] = {"ms_per_game": 1e3 * dt / n_games, "us_per_ply": 1e6 * dt / plies, "games_per_s": n_games / dt}
    if refshim.available():
        rb = refshim.load().board
        t0 = time.perf_counter()
        ref = [play_a_game_through(rb, 7, g, mg) for g in range(n_games)]
        dt = time.perf_counter() - t0
        out["reference_board_py"] = {"ms_per_game": 1e3 * dt / n_games, "us_per_ply": 1e6 * dt / plies,
                                     "games_per_s": n_games / dt, "cores": 1}
        out["identical_games"] = got == ref
        out["facade_speedup"] = out["reference_board_py"]["ms_per_game"] / out["b200_facade"]["ms_per_game"]
    return out


def cpu_baseline(budget_s=12.0, max_games_per_worker=1 << 30, seed=1, full_path_s=0.0):
    """reference CPU path on all host cores for ~budget_s seconds (+ full_path_s seconds of the
    play_a_turn-equivalent path, reported separately)."""
    import multiprocessing as mp
    from oracle import refshim
    kind = "reference" if refshim.available() else "port"
    if kind == "port":
        from oracle import lib as orc
        orc.build()
    cores = os.cpu_count() or 1
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(kind, seed, w * (1 << 24), budget_s, max_games_per_worker) for w in range(cores)])
    dt = time.perf_counter() - t0
    plies = sum(r[0] for r in res)
    games = sum(r[1] for r in res)
    what = ("reference board.py (oracle/_ref py3 transcription)" if kind == "reference"
            else "oracle/othello_oracle.c port (reference not present on this box)")
    extra = {}
    if kind == "reference" and full_path_s > 0:
        t1 = time.perf_counter()
        with ctx.Pool(cores) as pool:
            res2 = pool.map(_cpu_worker, [("reference_full", seed, w * (1 << 24), full_path_s, max_games_per_worker)
                                          for w in range(cores)])
        dt2 = time.perf_counter() - t1
        extra = {"full_play_a_turn_path": {"value": sum(r[0] for r in res2) / dt2, "unit": UNIT,
                                           "games_per_s": sum(r[1] for r in res2) / dt2,
                                           "what": "adds str(board), recorder-style serialisation and its "
                                                   "is_game_over per ply (game_runner.py:154-163, "
                                                   "game_recorder.py:107-114), %.1f s" % dt2}}
    return {"value": plies / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "games_per_s": games / dt, **extra,
            "sample": "%d random-playout games (%d plies) from the standard opening, bare loop "
                      "puttables->choose->put_s->is_game_over, %s, multiprocessing.Pool(%d), %.1f s"
                      % (games, plies, what, cores, dt)}, dt


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # each step = a bounded sample of the workload; whole run stays within a few minutes
    per_step = args.cpu_seconds if args.cpu_seconds else max(2.0, min(20.0, 90.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_baseline(budget_s=min(per_step, 3.0))
    total_plies = total_games = 0.0
    total_dt = 0.0
    last = None
    for _ in range(args.steps):
        last, dt = cpu_baseline(budget_s=per_step)
        total_plies += last["value"] * dt
        total_games += last["games_per_s"] * dt
        total_dt += dt
    value = total_plies / total_dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "games_per_s": total_games / total_dt,
        "config": {"workload": "config3_random_playout", "games_per_gpu": args.games, "t_max": T_MAX,
                   "note": "each step is a %.0f s time-bounded sample of the same workload on all host cores" % per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": last["kind"],
                         "sample": last["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# host-side placement of a rank
# ------------------------------------------------------------------------------------------------
def bind_rank_to_cores(local, world):
    """Give every rank of a node its own contiguous share of the cores this process may run on, so the
    submission threads of N ranks (and their pinned buffers, first-touched from those cores) do not
    migrate over each other.  Returns what was done, for the JSON line."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // max(1, world))
        mine = cores[local * per:(local + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return {"cores": "%d-%d" % (mine[0], mine[-1]), "n": len(mine), "of": len(cores)}
    except (AttributeError, OSError) as e:           # pragma: no cover - platform without sched_setaffinity
        return {"error": str(e)}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """samples SM clock and throttle reasons through NVML in a thread WHILE the timed region runs
    (the region lasts tens of ms, too short for `nvidia-smi -lms`); same fields as the recipe's
    nvidia-smi line: clocks.sm, clocks.max.sm, clocks_event_reasons.*"""

    def __init__(self, cuda_index):
        self.cuda_index = cuda_index
        self.samples = []
        self.reasons = 0
        self.max_mhz = None
        self.handle = None
        self.err = None
        self._stop = threading.Event()
        self.thread = None

    def start(self):
        try:
            import pynvml
            import torch
            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(self.cuda_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.cuda_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self._sample()
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception as e:                       # pragma: no cover - depends on the box
            self.err = "%s: %s" % (type(e).__name__, e)
            self.handle = None

    def _sample(self):
        nv = self.nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
        self.reasons |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))

    def _pump(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                break
            time.sleep(0.001)

    def stop(self):
        if self.handle is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        self._stop.set()
        self.thread.join(timeout=2)
        nv = self.nv
        names = [("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                 ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                 ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap),
                 ("hw_power_brake", nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown)]
        reasons = [n for n, bit in names if self.reasons & bit]
        sm = sorted(self.samples[1:] or self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm), "how": "NVML SM clock + throttle reasons polled every ~1 ms during the timed region"}


# ------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def config4_extra(dev, rank, world, G=1 << 19, reps=5, random_plies=10):
    """BASELINE config 4 under the driver: greedy self-play with the default_value() rows
    (parameter_progress_position_moves_learn.py:30-36), G games per GPU, first `random_plies` plies
    uniform-random (N_RAND_HAND_UNTIL, game_runner.py:6), full trajectories.  Device-timed, max over ranks."""
    import torch
    import torch.distributed as dist
    from subproc_b200 import ops, parameter
    w = torch.from_numpy(parameter.ProgressPositionMovesParameter().weights_table()).to(dev)
    pg = ops.playout(G, seed=2, gid0=rank * G, device=dev, policy=ops.POLICY_GREEDY, random_plies=random_plies, weights=w)
    tot = torch.zeros(4, dtype=torch.int64, device=dev)
    for i in range(2):
        ops.playout(G, seed=2, gid0=(world * (1 + i) + rank) * G, device=dev, policy=ops.POLICY_GREEDY,
                    random_plies=random_plies, weights=w, out=pg)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        ops.playout(G, seed=2, gid0=(world * (3 + i) + rank) * G, device=dev, policy=ops.POLICY_GREEDY,
                    random_plies=random_plies, weights=w, out=pg, totals=tot)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    # children evaluated by the last launch: sum of mobility over the plies the greedy engine searched
    children = torch.zeros((), dtype=torch.int64, device=dev)
    zero = torch.zeros(G, dtype=torch.int64, device=dev)
    for t in range(random_plies, int(pg.nplies.max().item())):
        own, opp = (pg.black[t], pg.white[t]) if t % 2 == 0 else (pg.white[t], pg.black[t])   # Black, White alternate strictly
        n = ops.counts(ops.legal(own, opp), zero)[:, 0].to(torch.int64)
        children += torch.where((pg.nplies > t) & (n > 1), n, torch.zeros_like(n)).sum()
    v = torch.tensor([float(tot[0]), float(G * reps), float(children) * reps], dtype=torch.float64, device=dev)
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    sec = float(tmax[0]) * 1e-3
    executed = None
    kp = os.path.join(ROOT, "profiles", "greedy_kernel_costs.json")
    if os.path.isfile(kp):
        kc = json.load(open(kp))
        rate = float(v[2]) / world / (sec * 1e3)                         # children per ms per GPU, this run
        executed = {"source": "profiles/greedy_kernel_costs.json (ncu --set full of one launch: %s)" % kc["source"],
                    "thread_inst_per_child": kc["thread_inst_per_child"], "active_lanes_per_inst": kc["active_lanes_per_inst"],
                    "alu_pipe_pct_ncu": kc["alu_pipe_pct"], "fmaheavy_pipe_pct_ncu": kc["fmaheavy_pipe_pct"],
                    "xu_pipe_pct_ncu": kc["xu_pipe_pct"], "issue_slot_pct_ncu": kc["issue_slot_pct"],
                    "alu_pipe_frac_at_this_runs_rate": kc["alu_pipe_pct"] / 100.0 * rate / kc["children_per_ms_under_ncu"],
                    "thread_inst_per_s": float(v[2]) / sec * kc["thread_inst_per_child"]}
    return {"workload": "config4_greedy_selfplay", "roofline": {"bound": "int32 ALU pipe", "executed": executed}, "games_per_gpu": G, "random_plies": random_plies, "launches": reps,
            "weights": "default_value() rows", "kernel_ms": float(tmax[0]) / reps,
            "positions_per_s": float(v[0]) / sec, "games_per_s": float(v[1]) / sec,
            "children_per_s": float(v[2]) / sec,
            "children_note": "successor positions evaluated (flip + move generation + 9-term evaluation each); counted "
                             "on the last launch and scaled by the number of launches",
            "black_minus_white_mean": float(tot[1]) / float(G * reps)}


def config5_extra(dev, rank, world, G=1 << 16, iters=10, warm=3, random_plies=10):
    """BASELINE config 5 under the driver: per iteration greedy self-play with the current weights ->
    exact integer statistics -> ONE all-reduce (NCCL) of 320 int64 -> four regressions on the device ->
    the next self-play reads the new table.  Replaces the Redis `fitting:*` polling
    (progress_position_moves_learn.py:112-158, parallel_learner_task.py:8-23).  Carries its own parity bits."""
    import torch
    import torch.distributed as dist
    from subproc_b200 import ops, parameter, learner
    w = torch.from_numpy(parameter.ProgressPositionMovesParameter().weights_table()).to(dev)
    acc = torch.zeros((4, learner.N_ACC), dtype=torch.int64, device=dev)
    stats = torch.empty((4, 112), dtype=torch.float64, device=dev)
    po = params = fits = acc_last = None
    ar = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w_used = None
    for it in range(warm + iters):
        if it == warm:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev0.record()
        if it == warm + iters - 1:
            w_used = w.clone()
        po = ops.playout(G, seed=3, gid0=(it * world + rank) * G, device=dev, policy=ops.POLICY_GREEDY,
                         random_plies=random_plies, weights=w, out=po)
        ops.learn_accumulate(po, acc=acc)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        learner.allreduce_stats(acc)
        a1.record()
        if it >= warm:
            ar.append((a0, a1))
        if it == warm + iters - 1:
            acc_last = acc.clone()                            # (the refit clears the accumulators)
        w, params, fits = ops.learn_refit(acc, w, weights_out=w, clear=True, params=params, fits=fits)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / iters
    ar_ms = sorted(a.elapsed_time(b) for a, b in ar)[len(ar) // 2]
    # parity: (1) the all-reduced accumulators of the last iteration == rank 0 replaying the union of the ranks'
    # game ids alone; (2) every rank ends with the same parameters
    same_acc = True
    if rank == 0:
        it = warm + iters - 1
        union = ops.playout(G * world, seed=3, gid0=it * world * G, device=dev, policy=ops.POLICY_GREEDY,
                            random_plies=random_plies, weights=w_used)
        same_acc = bool(torch.equal(ops.learn_accumulate(union), acc_last))
        del union
    same_params = True
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        gathered = [torch.empty_like(params) for _ in range(world)]
        dist.all_gather(gathered, params)
        same_params = all(bool(torch.equal(g, params)) for g in gathered)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    return {"workload": "config5_parallel_learner", "games_per_gpu_per_iteration": G, "iterations": iters,
            "iteration_ms": ms, "games_per_s": G * world / (ms * 1e-3), "allreduce_ms": ar_ms if world > 1 else None,
            "allreduce_bytes": 4 * learner.N_ACC * 8, "nranks": world,
            "launches_per_iteration": "greedy_kernel, learn_kernel, [ncclAllReduce], refit_kernel",
            "parity": {"allreduced_accumulators_equal_rank0_replay_of_all_game_ids": same_acc,
                       "parameters_identical_on_all_ranks": same_params},
            "parameters": [int(v) for v in params.cpu().tolist()],
            "fit": "normal equations over every (position, side) sample of the iteration; the reference instead fits "
                   "each shard on <= 50 000 keys sampled from its smoothed value table "
                   "(progress_position_moves_learn.py:66-86,160-184) -- that path is subproc_b200.value_table"}


def config5_table_extra(dev, G=1 << 16, iters=3, warm=1, random_plies=10):
    """The same iteration with the REFERENCE's learning semantics (single GPU): every (position, side) of the greedy
    games smooths the order-dependent value table in the reference's update order
    (progress_position_moves_learn.py:37-62), then each shard is refitted on <= 50 000 distinct sampled table entries
    (:66-86,160-184) and stored with int() truncation (:196-209).  Wall clock, synchronised per iteration."""
    import torch
    from subproc_b200 import learner
    L = learner.ProgressPositionMovesLearn()
    L.configure({})
    times, nsamples, params = [], None, None
    for it in range(warm + iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _po, (_mses, _scores, params, nsamples) = L.self_play_iteration_table(G, seed=5, iteration=it,
                                                                           random_plies=random_plies, device=dev)
        torch.cuda.synchronize()
        if it >= warm:
            times.append(time.perf_counter() - t0)
    ms = 1e3 * min(times)
    return {"workload": "config5 with the reference's value-table semantics, one GPU", "games_per_iteration": G,
            "iterations": iters, "iteration_ms": ms, "games_per_s": G / (ms * 1e-3), "table_keys": len(L.table),
            "samples_per_shard": [int(v) for v in nsamples], "parameters": [int(v) for v in L.read_parameters()[1:]],
            "what": "greedy self-play -> (key, target) records in update order -> stable radix sort -> runs of equal keys "
                    "folded sequentially into the hash table in HBM (V = new if V == 0 else V * 0.97 + new * 0.03, fp64, "
                    "bit-identical to the reference loop) -> four fits on sampled table entries"}


DUMP_GAMES = 1 << 18          # --dump-outputs: games of the last timed step whose per-game results are written
DUMP_TRAJ_GAMES = 1 << 12     # ... and how many of them also have their whole trajectory written (28 MB in all)


def _bits_halves(a):
    """int64 bit patterns -> float64 [..., 2] (low, high 32-bit halves): exact, where one float64 would round"""
    import numpy as np
    u = a.view(np.uint64)
    return np.stack([u & 0xFFFFFFFF, u >> 32], axis=-1).astype(np.float64)


def sample_outputs(po, gid0, totals):
    """What the caller of one ops.playout launch receives, on a fixed seeded sample of its games (game ids from gid0):
    nplies and final positions of DUMP_GAMES games, trajectories of DUMP_TRAJ_GAMES of them.  Bitboards are (low, high)
    halves; trajectory entries past a game's end, which the kernel leaves unspecified, are -1.  ``totals`` (int64 [4]:
    plies, sum of n_black - n_white, Black wins, White wins) is written as it stands."""
    import numpy as np
    import torch
    rng = np.random.default_rng(0)
    T = po.t_max
    idx = np.sort(rng.choice(po.n_games, size=min(po.n_games, DUMP_GAMES), replace=False))
    tix = np.sort(rng.choice(idx, size=min(idx.size, DUMP_TRAJ_GAMES), replace=False))
    nplies = po.nplies.cpu().numpy()
    sel = torch.from_numpy(tix).to(po.nplies.device)
    tb = _bits_halves(po.black.index_select(1, sel).cpu().numpy())           # [T+1][n][2]
    tw = _bits_halves(po.white.index_select(1, sel).cpu().numpy())
    tm = po.move.index_select(1, sel).cpu().numpy().astype(np.float32)       # [T][n]
    t = np.arange(T + 1)[:, None]
    end = np.minimum(nplies[tix], T)[None, :]
    tb[t > end] = -1
    tw[t > end] = -1
    tm[t[:-1] >= end] = -1
    return {"game_id": (gid0 + idx).astype(np.float64), "nplies": nplies[idx].astype(np.float32),
            "final_black": _bits_halves(po.final_black.cpu().numpy()[idx]),
            "final_white": _bits_halves(po.final_white.cpu().numpy()[idx]),
            "trajectory_game_id": (gid0 + tix).astype(np.float64),
            "trajectory_black": tb, "trajectory_white": tw, "trajectory_move": tm,
            "totals": totals.cpu().numpy().astype(np.float64)}


def run_b200_arm(args):
    import ctypes
    import torch
    import torch.distributed as dist
    from subproc_b200 import ops, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path is sm_100a kernels, there is no CPU fallback")
    cb = None
    if world == 1 and not args.no_cpu_baseline:
        secs = args.cpu_seconds if args.cpu_seconds else 12.0
        cb, _ = cpu_baseline(budget_s=secs, full_path_s=secs / 2)          # before CUDA is initialised (fork-safe)
    # host side of a rank: its own cores, one intra-op thread (the only torch CPU work left is scalars)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    binding = bind_rank_to_cores(local, local_world) if local_world > 1 else None
    torch.set_num_threads(1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    G = args.games
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: value ---------------------------------------------------------
    # K launches of G games each.  Consecutive launches alternate over two streams (each with its own 2 GB
    # trajectory buffer), so the thinning tail of one launch runs under the head of the next -- what any
    # caller that streams batches does, and what the host-buffer path below does with its chunks.
    streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
    pos = [ops.playout(G, seed=1, gid0=0, device=dev, t_max=T_MAX) for _ in range(2)]
    tot = [torch.zeros(4, dtype=torch.int64, device=dev) for _ in range(2)]
    po = pos[0]
    gid_base = rank * (W + K) * G * 2

    def one_step(i, count):
        k = i % 2
        with torch.cuda.stream(streams[k]):
            ops.playout(G, seed=1, gid0=gid_base + i * G, device=dev, t_max=T_MAX, out=pos[k],
                        totals=tot[k] if count else None)

    torch.cuda.synchronize()
    for i in range(W):
        one_step(i, False)
    torch.cuda.synchronize()
    int_peak_alu = ops.int32_peak(dev)                                     # ALU pipe alone (LOP3/SHF), lane-ops/s
    int_peak = ops.int32_peak(dev, dual=True)                              # ALU + FMA pipes (LOP3 + IMAD): the integer ceiling
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    cur = torch.cuda.current_stream(dev)
    ev_start, ev_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev_start.record(cur)
    for st in streams:
        st.wait_event(ev_start)
    for i in range(K):
        one_step(W + i, True)
        evs[i].record(streams[i % 2])
    for st in streams:
        cur.wait_stream(st)
    ev_end.record(cur)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    # taken now: the launches timed alone below reuse the buffers of the timed steps.  The totals, from which `value`
    # is computed, are those of all K timed steps (each stream accumulates its own).
    i_last = W + K - 1
    outputs = (sample_outputs(pos[i_last % 2], gid_base + i_last * G, tot[0] + tot[1])
               if args.dump_outputs and rank == 0 else None)
    # time a launch spends in its stream (launches of the two streams overlap, so these add up to more than the total)
    step_ms = [(ev_start if i < 2 else evs[i - 2]).elapsed_time(evs[i]) for i in range(K)]
    total_ms = ev_start.elapsed_time(ev_end)
    positions = int(tot[0][0].item()) + int(tot[1][0].item())
    games = K * G
    # one launch alone (nothing else on the GPU): the duration the ncu launch list is compared with
    alone_ms = []
    for i in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        ops.playout(G, seed=1, gid0=gid_base + (W + K + i) * G, device=dev, t_max=T_MAX, out=po)
        e1.record()
        e1.synchronize()
        alone_ms.append(e0.elapsed_time(e1))

    # ---- the batch API on explicit positions: othello_step (put_s + game-over check) on synthetic
    # random-opening positions = the positions of this launch after 10 random plies, their next move
    t_open = 10
    sb, sw = po.black[t_open].clone(), po.white[t_open].clone()
    mv = po.move[t_open].contiguous()
    wb, ww = torch.empty_like(sb), torch.empty_like(sw)
    turn = torch.empty(G, dtype=torch.uint8, device=dev)
    nturn = torch.empty(G, dtype=torch.int32, device=dev)
    fl, rt, fg = torch.empty_like(sb), torch.empty(G, dtype=torch.int32, device=dev), torch.empty(G, dtype=torch.uint8, device=dev)
    step_times = []
    for i in range(3 + 5):
        wb.copy_(sb); ww.copy_(sw); turn.fill_(ops.BLACK); nturn.fill_(t_open)      # restore (untimed)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.step(wb, ww, turn, nturn, mv, fl, rt, fg)
        e1.record()
        e1.synchronize()
        if i >= 3:
            step_times.append(e0.elapsed_time(e1))
    step_live = int((rt > 0).sum().item())
    step_info = {"positions_per_s": G / (min(step_times) * 1e-3), "kernel_ms": min(step_times), "positions": G,
                 "legal_moves_applied": step_live,
                 "what": "othello_step (put_s + pass / game-over flags) on the positions after %d random plies; "
                         "50 B of HBM traffic per position" % t_open}

    # ---- end-to-end arm: host buffers through the C ABI ---------------------------------------
    # The call a user without torch makes (INTEGRATION.md): start positions in pinned host memory go in
    # (16 B per game), the per-game results come back to pinned host memory as two-byte summaries (plies,
    # disc difference: what store_batch_stats reads of a game, learn_base.py:70-98) together with the batch
    # totals, every step.  Two batches are kept in flight (othello_playout_host_async / othello_ctx_wait), so
    # the PCIe copies of one step run under the kernels of its neighbours; the timed region still starts with
    # nothing in flight and ends when the last result of step K is in host memory.  (The full 20 B per game --
    # plies as int32 + the final position -- is measured next to it: on an 8-GPU host the PCIe fabric, not the
    # GPUs, then sets the pace, see profiles/e2e_breakdown_r02_*.json.)
    L = _lib.lib()
    ctx = ctypes.c_void_p()
    _lib.check(L.othello_ctx_create(local, ctypes.byref(ctx)), "othello_ctx_create")
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
    h_b0 = pin(G, torch.int64).fill_(ops.signed64(ops.START_BLACK))
    h_w0 = pin(G, torch.int64).fill_(ops.signed64(ops.START_WHITE))
    h_out = [(pin(G, torch.int16), pin(4, torch.int64), pin(G, torch.int32), pin(G, torch.int64), pin(G, torch.int64))
             for _ in range(2)]
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    e2e_gid = [gid_base + (W + K + 3) * G]

    def e2e_run(steps, full=False, upload=True):
        """issue step i+1, then collect step i; returns the positions played (from the batch totals)"""
        tickets = [0, 0]
        played = 0
        for i in range(steps + 1):
            if i < steps:
                o = h_out[i % 2]
                tk = ctypes.c_int64()
                _lib.check(L.othello_playout_host_async(
                    ctx, 1, e2e_gid[0], G, P(h_b0) if upload else None, P(h_w0) if upload else None, None,
                    ops.POLICY_RANDOM, 0, 0, 0, None, -1, None, T_MAX,
                    None, None, None, P(o[2]) if full else None, P(o[3]) if full else None, P(o[4]) if full else None,
                    None if full else P(o[0]), P(o[1]), ctypes.byref(tk)), "othello_playout_host_async")
                e2e_gid[0] += G
                tickets[i % 2] = tk.value
            if i > 0:
                _lib.check(L.othello_ctx_wait(ctx, tickets[(i - 1) % 2]), "othello_ctx_wait")
                played += int(h_out[(i - 1) % 2][1][0])                  # the step's result, read on the host
        return played

    def e2e_timed(full, upload=True):
        e2e_run(max(3, min(W, 5)), full, upload)
        barrier()
        t0 = time.perf_counter()
        played = e2e_run(K, full, upload)
        torch.cuda.synchronize()
        return played, time.perf_counter() - t0

    e2e_positions, e2e_s = e2e_timed(False)
    # untimed check of the last batch: the per-game summaries on the host agree with the device-side totals
    last = h_out[(K - 1) % 2]
    sm = last[0].numpy().view("uint16")
    e2e_ok = (int((sm & 0xff).sum()) == int(last[1][0]) and
              int((sm >> 8).astype("uint8").view("int8").sum()) == int(last[1][1]) and int((sm & 0xff).min()) > 0)
    full_positions, full_s = e2e_timed(True)                             # 20 B per game back instead of 2
    e2e_ok = e2e_ok and int(last[2].sum(dtype=torch.int64)) == int(last[1][0])
    # what GameRunner.play_a_game itself does (game_runner.py:165-170: every game starts from a fresh Board()): no start
    # positions to upload (NULL = the standard opening), two-byte summaries + totals back
    std_positions, std_s = e2e_timed(False, upload=False)
    # a single synchronous call (copy-in, kernels, copy-out, wait): the latency of one batch
    sync_ms = []
    for i in range(5):
        t1 = time.perf_counter()
        _lib.check(L.othello_playout_host(ctx, 1, e2e_gid[0], G, P(h_b0), P(h_w0), None, ops.POLICY_RANDOM, 0, 0, 0, None,
                                          -1, None, T_MAX, None, None, None, P(last[2]), P(last[3]), P(last[4])),
                   "othello_playout_host")
        sync_ms.append(1e3 * (time.perf_counter() - t1))
        e2e_gid[0] += G
    L.othello_ctx_destroy(ctx)
    h2d = G * (8 + 8)
    d2h = G * 2 + 32

    # ---- the other two GPU workloads of BASELINE.json, each with its own figures ------------------
    extra = {}
    if not args.no_extra:
        extra["config4"] = config4_extra(dev, rank, world)
        extra["config5"] = config5_extra(dev, rank, world)
        if world == 1:
            extra["config5_table"] = config5_table_extra(dev)

    # ---- reduce over ranks -----------------------------------------------------------------------
    if world > 1:
        t = torch.tensor([total_ms, e2e_s * 1e3, full_s * 1e3, std_s * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c = torch.tensor([positions, games, e2e_positions, full_positions, std_positions], dtype=torch.float64, device=dev)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        total_ms, e2e_ms, full_ms, std_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        positions, games, e2e_positions, full_positions, std_positions = (float(c[i]) for i in range(5))
    else:
        e2e_ms, full_ms, std_ms = e2e_s * 1e3, full_s * 1e3, std_s * 1e3

    if rank == 0:
        value = positions / (total_ms * 1e-3)
        hbm_peak, hbm_src = measured_peaks()
        # the dominant (only) kernel of a step is playout_kernel<traj, uniform>; with two launches in flight the
        # time a launch costs is the timed region divided by the launches in it
        kern_ms = total_ms / K
        pos_per_launch = positions / (K * n_gpus)
        achieved_ops = pos_per_launch * LANE_OPS_PER_POSITION / (kern_ms * 1e-3)
        achieved_gbs = pos_per_launch * BYTES_PER_POSITION / (kern_ms * 1e-3) / 1e9
        # what ncu measured on one launch of this kernel (profiles/playout_kernel_costs.json, written by
        # tools/kernel_costs.py from the committed ncu summary): DRAM traffic, executed instructions, pipe utilisation
        traffic, executed = None, None
        tp = os.path.join(ROOT, "profiles", "playout_kernel_costs.json")
        if os.path.isfile(tp):
            kc = json.load(open(tp))
            traffic = kc.get("dram_bytes_per_launch")
            live_rate = pos_per_launch / kern_ms                       # positions per ms, this run
            scale = live_rate / kc["positions_per_ms_under_ncu"]
            executed = {
                "source": "profiles/playout_kernel_costs.json (ncu --set full of one launch: %s)" % kc["source"],
                "thread_inst_per_position": kc["thread_inst_per_position"],
                "active_lanes_per_inst": kc["active_lanes_per_inst"],
                "alu_pipe_pct_ncu": kc["alu_pipe_pct"], "fmaheavy_pipe_pct_ncu": kc["fmaheavy_pipe_pct"],
                "xu_pipe_pct_ncu": kc["xu_pipe_pct"], "issue_slot_pct_ncu": kc["issue_slot_pct"],
                "alu_pipe_frac_at_this_runs_rate": kc["alu_pipe_pct"] / 100.0 * scale,
                "note": "utilisation of the binding pipe (integer ALU) = the ncu figure scaled by this run's "
                        "positions/s over the profiled launch's (the instructions per position are a constant of the kernel)"}
        # roofline.frac: a utilisation.  The kernel is bound by instruction issue (one warp instruction per clock per
        # SM sub-partition, which is also what LOP3 + IMAD co-issue reaches: the measured peak) with the ALU pipe as the
        # busiest pipe behind it.  achieved = executed thread instructions per second = positions/s x the kernel's
        # executed thread instructions per position (ncu, a constant of the kernel).
        if executed is not None:
            roof_achieved = value / n_gpus * executed["thread_inst_per_position"]
            roof_unit = "Tthread-inst/s"
            roof_def = ("utilisation of the instruction issue rate: positions/s x executed thread instructions per position "
                        "(ncu smsp__inst_executed x active lanes / positions of one launch, profiles/playout_kernel_costs.json) "
                        "over the measured peak of 32-bit integer instruction issue (LOP3 + IMAD co-issued, csrc/peak.cu, "
                        "measured in this run; 148 SMs x 128 lanes x clock in theory); per GPU")
        else:
            roof_achieved, roof_unit = achieved_ops, "Tlane-op/s"
            roof_def = "algorithm-normalised (profiles/playout_kernel_costs.json missing): see algorithmic_definition"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "games_per_s": games / (total_ms * 1e-3),
            "config": {"workload": "config3_random_playout", "games_per_gpu": G, "t_max": T_MAX,
                       "policy": "uniform random, standard opening, seed 1",
                       "trajectory": "full SoA [t][game] black,white u64 + move u8 in HBM",
                       "l2": "kernel reads no input from HBM; ~%.2f GB written per step exceeds the 126 MB L2"
                             % (pos_per_launch * BYTES_PER_POSITION / 1e9),
                       "parallelism": "games sharded over %d GPU(s), no data-path collective" % n_gpus},
            "roofline": {"bound": "int32", "achieved": roof_achieved / 1e12, "peak": int_peak / 1e12,
                         "unit": roof_unit, "frac": roof_achieved / int_peak, "traffic": traffic,
                         "frac_definition": roof_def,
                         "algorithmic_achieved": achieved_ops / 1e12, "algorithmic_frac": achieved_ops / int_peak,
                         "algorithmic_definition": "positions/s x the canonical 512 lane-ops of 8-direction Kogge-Stone "
                                                   "(SURVEY.md 8d) over the same peak: ALGORITHM-normalised throughput, not "
                                                   "a utilisation (above 1 since put() became four table look-ups: the "
                                                   "kernel executes ~330 instructions per position, 152 of them on the ALU pipe)",
                         "executed": executed,
                         "peak_source": "csrc/peak.cu, measured in this run: LOP3 + IMAD co-issued on the ALU and FMA "
                                        "pipes (the two pipes that execute 32-bit integer lane-ops)",
                         "peak_alu_pipe_only": int_peak_alu / 1e12,
                         "algorithmic": "%d INT32 lane-ops per position-step (SURVEY.md 8d)" % LANE_OPS_PER_POSITION,
                         "kernel": "playout_kernel<random,traj>", "kernel_ms": kern_ms,
                         "kernel_ms_definition": "timed region / launches (consecutive launches alternate over two "
                                                 "streams); a launch alone on the GPU takes kernel_alone_ms, and "
                                                 "spends kernel_in_stream_ms in its stream when two are in flight",
                         "kernel_alone_ms": min(alone_ms), "kernel_in_stream_ms": sum(step_ms) / K,
                         "hbm": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": achieved_gbs / hbm_peak, "peak_source": hbm_src,
                                 "algorithmic": "%d B written per position" % BYTES_PER_POSITION}},
            "e2e": {"value": e2e_positions / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "games_per_s": G * K * n_gpus / (e2e_ms * 1e-3),
                    "ms_per_step": e2e_ms / K, "frac_of_value": (e2e_positions / e2e_ms) / (positions / total_ms),
                    "sync_call_ms": min(sync_ms), "results_checked": bool(e2e_ok), "host_binding": binding,
                    "full_results": {"value": full_positions / (full_ms * 1e-3), "unit": UNIT,
                                     "d2h_bytes_per_step": G * 20 + 32,
                                     "what": "the same with plies (int32) + final position (2 x u64) per game instead "
                                             "of the two-byte summary"},
                    "standard_opening": {"value": std_positions / (std_ms * 1e-3), "unit": UNIT,
                                         "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h,
                                         "what": "the same without the upload: start positions NULL = every game from "
                                                 "the standard opening, as GameRunner.play_a_game does "
                                                 "(game_runner.py:165-170); on an 8-GPU host whose PCIe fabric gives "
                                                 "each GPU ~24 GB/s the 16 B per game of the headline cost ~0.7 ms per "
                                                 "step next to a ~0.73 ms kernel"},
                    "api": "othello_playout_host_async + othello_ctx_wait (C ABI, pinned host buffers, two batches "
                           "in flight; start positions uploaded (16 B per game), two-byte per-game summaries + batch "
                           "totals downloaded every step; trajectories stay in HBM); sync_call_ms = one synchronous "
                           "othello_playout_host call returning the full 20 B per game"},
            "gpu_launches": K,
            "step_kernel": step_info,
            "extra": extra,
            "clocks": clocks,
        }
        if cb is not None:
            cb["config1_single_game_facade"] = config1_facade()
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    if outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=1 << 20, help="games per GPU per step")
    ap.add_argument("--cpu-seconds", type=float, default=None,
                    help="seconds of host-core time per CPU sample (default: 12 for the cpu_baseline leg, "
                         "90 / (steps + warmup) clamped to [2, 20] per step of --impl reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 4 / config 5 objects")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (a fixed sample of its games, rank "
                         "0's with several GPUs) and the totals of all of them as DIR/<name>.npy in float32 / float64, "
                         "for comparing two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3                      # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
