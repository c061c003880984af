/*
 * othello_b200.h -- C ABI of the B200-native batched Othello hot path.
 *
 * This is the drop-in boundary for the rules / step-loop / feature / evaluation / learner-
 * statistics path of ysnrkdm/subproc.  The reference has no native code, so there is no
 * existing FFI to mirror; each entry point instead names the reference function it replaces
 * (file:line in the reference tree).  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - bitboards: uint64, bit s = x + 8*y, x = file a..h = 0..7, y = rank 1..8 = 0..7
 *     (the mask convention of board.py:79 and coord_from_handstr board.py:176-185);
 *   - colours: 0 Empty, 1 Black, 2 White (board.py:3-7); Black moves first (board.py:26);
 *   - moves: uint8 square 0..63, 64 = pass ('ps'/'PS', board.py:194), anything else is a hand
 *     string that does not parse (put_s returns -1);
 *   - "_host" functions take HOST pointers and run on the context's own stream and workspace;
 *     all others take DEVICE pointers, launch asynchronously on `stream` (a cudaStream_t passed
 *     as void*), allocate nothing and keep no global state -- except othello_playout with the
 *     random engine, which keeps its opening book on the device (see there);
 *   - every function returns 0 on success, a positive cudaError_t value, or a negative
 *     OTHELLO_E_* code.  othello_error_string() explains both.
 */
#ifndef OTHELLO_B200_H
#define OTHELLO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OTHELLO_ABI_VERSION 4

#define OTHELLO_EMPTY 0
#define OTHELLO_BLACK 1
#define OTHELLO_WHITE 2
#define OTHELLO_PASS  64

#define OTHELLO_START_BLACK 0x0000000810000000ull   /* board.py:25 */
#define OTHELLO_START_WHITE 0x0000001008000000ull   /* board.py:24 */

#define OTHELLO_E_INVALID   (-1)   /* bad argument (null pointer, negative size, depth out of range) */
#define OTHELLO_E_WORKSPACE (-2)   /* caller-supplied workspace too small */
#define OTHELLO_E_NO_DEVICE (-3)   /* no CUDA device / driver */

/* step flags (othello_step `flags`, describing the position AFTER the move) */
#define OTHELLO_F_MUST_PASS 1      /* side to move has no move but the game is not over */
#define OTHELLO_F_GAME_OVER 2      /* Board.is_game_over(), board.py:57-58 */

/* playout policies: what the two engines behind GameRunner answer to 'go' */
#define OTHELLO_POLICY_RANDOM 0    /* uniform over puttables(), 'ps' when empty */
#define OTHELLO_POLICY_GREEDY 1    /* arg-max of the linear evaluation of the successor, ties -> lowest square */

#define OTHELLO_FEATURES   10      /* counts(): discs, mobility, a..h (parameter_progress_position_moves_learn.py:5-17) */
#define OTHELLO_PHASES      4      /* disc-count shards (0,16),(17,32),(33,48),(49,64) (progress_position_moves_learn.py:112-113) */
#define OTHELLO_WEIGHTS    10      /* per phase: 9 weights over (mobility, a..h) + intercept */
#define OTHELLO_STATS     112      /* per phase: XtX[10][10], Xty[10], n, sum y^2 */

int         othello_abi_version(void);
const char *othello_error_string(int code);

/* ---- rules ---------------------------------------------------------------------------------- */

/* Board.puttables(piece) as a mask (board.py:46-52, via is_puttable_at :141-149 and
 * hands_for_direc :124-139).  own/opp: discs of `piece` / of the other colour. */
int othello_legal(const uint64_t *own, const uint64_t *opp, uint64_t *legal, int64_t n, void *stream);

/* Board.put(piece, x, y) without mutation (board.py:161-174): the set of discs that placing
 * `piece` on `square` flips; 0 when the square is occupied or nothing flips (put returns 0). */
int othello_flips(const uint64_t *own, const uint64_t *opp, const uint8_t *square, uint64_t *flips,
                  int64_t n, void *stream);

/* Board.put_s(hand) for the side to move, in place (board.py:192-209), plus the two
 * is_game_over()/pass checks play_a_turn and the recorders make after it (game_runner.py:162,
 * game_recorder.py:112).  ret: -1 illegal (state untouched), 0 pass, else number flipped.
 * flips_out, ret, flags may be NULL. */
int othello_step(uint64_t *black, uint64_t *white, uint8_t *turn, int32_t *nturn, const uint8_t *move,
                 uint64_t *flips_out, int32_t *ret, uint8_t *flags, int64_t n, void *stream);

/* n_black / n_white / n_empty (board.py:37-44): out[n][3] */
int othello_counts(const uint64_t *black, const uint64_t *white, int32_t *out, int64_t n, void *stream);

/* Board.mask_count(color, mask) (board.py:74-81): out[i] = popcount(discs of color[i] & mask[i]) */
int othello_mask_count(const uint64_t *black, const uint64_t *white, const uint8_t *color, const uint64_t *mask,
                       int32_t *out, int64_t n, void *stream);

/* Board.serialize_board / Board.deserialize (board.py:223-262): the 64-character row-major board
 * string of the recorder schema ('O' = Black, 'X' = White, '-' = empty; game_recorder.py:108-113).
 * chars: DEVICE char[n][64], 16-byte aligned.  Any other character deserialises to an empty square. */
int othello_serialize_boards(const uint64_t *black, const uint64_t *white, char *chars, int64_t n, void *stream);
int othello_deserialize_boards(const char *chars, uint64_t *black, uint64_t *white, int64_t n, void *stream);

/* ---- features and evaluation ---------------------------------------------------------------- */

/* counts(a_book, side) (parameter_progress_position_moves_learn.py:5-17): out[n][10] =
 * (64 - empties, mobility(side), popc(side & a) .. popc(side & h)); side = colour 1/2. */
int othello_features(const uint64_t *black, const uint64_t *white, const uint8_t *side, int32_t *out,
                     int64_t n, void *stream);

/* Linear phase-weighted evaluation (rows of default_value(),
 * parameter_progress_position_moves_learn.py:30-36; phase shards progress_position_moves_learn.py:112-113;
 * the form lr.predict evaluates at :178): out[i] = W[phase][0..8] . (mobility, a..h) + W[phase][9].
 * weights: DEVICE float[4][10]. */
int othello_eval(const uint64_t *black, const uint64_t *white, const uint8_t *side, const float *weights,
                 float *out, int64_t n, void *stream);

/* ---- the game-runner step loop -------------------------------------------------------------- */

/* GameRunner.play_a_game (game_runner.py:165-201) for n_games independent games, one launch.
 * Game g uses the counter-based RNG stream (seed, gid0 + g); results do not depend on how games
 * are sharded over launches or GPUs. */
typedef struct {
    uint64_t seed;
    uint64_t gid0;
    int64_t  n_games;
    const uint64_t *black0;       /* [n] initial positions, or NULL for the standard opening (board.py:22-27) */
    const uint64_t *white0;
    const uint8_t  *turn0;        /* [n] side to move, or NULL = Black */
    int32_t  policy;              /* OTHELLO_POLICY_* : the engine behind both players */
    int32_t  random_plies;        /* greedy engine answers uniformly at random while ply < random_plies */
    int32_t  n_rand_black;        /* go_for's substitution budget n_rand_hands (game_runner.py:116-119,133-152) */
    int32_t  n_rand_white;
    const float *weights;         /* DEVICE float[4][10]; required for OTHELLO_POLICY_GREEDY */
    int32_t  t_max;               /* trajectory capacity in plies (120 holds every game from <= 60 empties) */
    int64_t  stride;              /* games per trajectory row (>= n_games); random engine: (t_max + 2) * stride < 2^32 */
    uint64_t *traj_black;         /* [t_max+1][stride] position before ply t (recorder.add, game_runner.py:170,159); NULL = none */
    uint64_t *traj_white;
    uint8_t  *traj_move;          /* [t_max][stride] move played at ply t (0..63, 64 = pass) */
    int32_t  *nplies;             /* [n] plies played, passes included (= nturn of the terminal position) */
    uint64_t *final_black;        /* [n] terminal position */
    uint64_t *final_white;
    /* proc_black / proc_white may be different engines (GameRunner.__init__, game_runner.py:107-123): */
    int32_t  policy_white;        /* White's engine, or -1 = the same as `policy` (which is then both players') */
    int32_t  games_per_warp;      /* greedy engine: games a warp plays, 8 / 16 / 32; anything else = chosen from n_games */
    const float *weights_white;   /* DEVICE float[4][10] for White's greedy engine, or NULL = `weights` */
    /* what GameRunner.play_a_game reports at the end of a game (game_runner.py:194-199) and
     * store_batch_stats sums over a batch (learn_base.py:70-88), accumulated (+=) over the games of
     * this launch: [0] plies played, [1] sum of (n_black - n_white) as two's complement, [2] games Black
     * won, [3] games White won.  DEVICE uint64[4] or NULL; the caller zeroes it. */
    unsigned long long *totals;
    /* the same per game, in two bytes: low byte = plies played (saturating at 255), high byte = n_black -
     * n_white as int8 -- all that store_batch_stats needs of a game (learn_base.py:70-98), and a tenth of
     * the bytes of nplies + the final position when results cross PCIe.  DEVICE uint16[n] or NULL. */
    uint16_t *summary;
} othello_playout_args;

/* Device memory kept by the library: the random engine takes the first 8 plies of games that start from the
 * standard opening with Black to move from an opening book (the game tree of those plies, 455 221 nodes).  The
 * first random-engine call on a device allocates 14.6 MB there, uploads the book synchronously (the host keeps its
 * 14.6 MB copy) and keeps it until the process exits.  A call on a stream that is being captured into a CUDA graph
 * does not upload it: its kernel plays those plies itself.  Results do not depend on either. */
int othello_playout(const othello_playout_args *args, void *stream);

/* ---- perft ---------------------------------------------------------------------------------- */

/* Legal-move enumeration to `depth` plies (pass = one ply, a game-over node = one leaf).  Expands
 * breadth-first on the device, then counts the frontier nodes depth-first in registers.  The host never
 * reads the frontier: a call is a fixed sequence of launches steered by a control block in the workspace.
 * workspace: DEVICE scratch, >= othello_perft_workspace_bytes(depth).
 *
 * othello_perft: synchronous, result is a HOST pointer; OTHELLO_E_WORKSPACE if a frontier did not fit.
 * othello_perft_async: only enqueues; result is a DEVICE uint64[2] = {nodes, 1 if the workspace was too
 * small}, valid in stream order.  part / nparts split the depth-first stage: the call counts the frontier
 * nodes whose position hashes to `part` (and, for part 0, the game-over leaves met while expanding), so the
 * sum of the nparts results is the node count -- one u64 all-reduce across GPUs (SURVEY.md 8e). */
int64_t othello_perft_workspace_bytes(int depth);
int othello_perft(uint64_t black, uint64_t white, int turn, int depth, void *workspace, int64_t workspace_bytes,
                  uint64_t *result, void *stream);
int othello_perft_async(uint64_t black, uint64_t white, int turn, int depth, int part, int nparts,
                        void *workspace, int64_t workspace_bytes, uint64_t *result, void *stream);

/* ---- exact endgame solver ------------------------------------------------------------------- */

/* The perfect-play value and best move of n positions, one lane per position (negamax, alpha-beta).
 *   value: own - opponent discs of the terminal position reached when both sides play perfectly, "own" = the side
 *          to move; the game ends when neither side can move (Board.is_game_over, board.py:57-58) and a pass is a
 *          ply.  Empty squares left at the end are NOT given to the winner: this is the reference's own scoring
 *          (winner by disc count, game_runner.py:194-199; learner target own - opp final discs,
 *          progress_position_moves_learn.py:55), not the Edax / WTHOR convention.  Range -64..64.
 *   move:  the lowest square (x + 8*y) among the moves that reach the value; OTHELLO_PASS when the side to move has
 *          no move but the game is not over (value = minus the value with the other side to move);
 *          OTHELLO_NO_MOVE when the game is over (value = the disc difference).
 *   A position with more than OTHELLO_SOLVE_MAX_EMPTIES empty squares, or with black & white != 0, gets value
 *   OTHELLO_SOLVE_REFUSED and move OTHELLO_NO_MOVE; the rest of the batch is solved normally.
 *   nodes: positions the search visited, per position (benchmarking only): a function of the position alone,
 *          whatever the batch around it.  May be NULL.
 * turn: [n] side to move (OTHELLO_BLACK, anything else = White), or NULL = Black.  Asynchronous on `stream`,
 * DEVICE pointers.  workspace: DEVICE scratch, >= othello_solve_workspace_bytes(); holds the work counter of the
 * persistent grid, which the call resets itself.  n = 0 is a no-op. */
#define OTHELLO_SOLVE_MAX_EMPTIES 24
#define OTHELLO_SOLVE_REFUSED   (-128)
#define OTHELLO_NO_MOVE          255
int64_t othello_solve_workspace_bytes(void);
int othello_solve(const uint64_t *black, const uint64_t *white, const uint8_t *turn, int32_t *value, uint8_t *move,
                  uint64_t *nodes, int64_t n, void *workspace, int64_t workspace_bytes, void *stream);

/* ---- learner sufficient statistics ---------------------------------------------------------- */

/* For every recorded position t of every game and both sides ('O' = Black then 'X' = White,
 * progress_position_moves_learn.py:44-47): x = (mobility, a..h, 1), y = (own - opp final discs) *
 * decay[nplies - t] (:55, decay[k] = 0.9 ** k computed by the host in fp64), accumulated (+=) per phase
 * shard into EXACT integer accumulators acc[4][OTHELLO_ACC] (DEVICE int64, caller zeroes):
 *   [0..54]  upper triangle of XtX[10][10], row-major (the sample count n is its last entry, 1 x 1);
 *   [56+2k], [57+2k]  high / low word of the 2^-40 fixed-point sum k: Xty[0..8] for k = 0..8, sum y^2 for k = 9
 *            (every game contributes its fp64 partial sums, formed in ply order, rounded once to 2^-40).
 * Integer sums do not depend on the order of additions: the accumulators -- and therefore the learnt
 * parameters -- are bit-identical however games are split over launches, ranks or GPUs, and the ranks'
 * exchange is an all-reduce(SUM) of these 320 int64.  Games with nplies > t_max are skipped. */
#define OTHELLO_ACC 80
int othello_learn_accumulate(const uint64_t *traj_black, const uint64_t *traj_white, const int32_t *nplies,
                             const uint64_t *final_black, const uint64_t *final_white,
                             int64_t n_games, int64_t stride, int32_t t_max, const double *decay /* [t_max+1] */,
                             int64_t *acc, void *stream);

/* acc[4][OTHELLO_ACC] -> stats[4][OTHELLO_STATS] doubles (=): XtX[10][10], Xty[10], n, sum y^2; every
 * value is the correctly rounded image of its exact integer sum.  DEVICE pointers. */
int othello_learn_stats(const int64_t *acc, double *stats, void *stream);

/* fit_parameter for the four shards ON the device (progress_position_moves_learn.py:160-184, minus
 * its sampling): OLS with intercept from stats[4][112] (minimum-norm when a shard is rank deficient),
 * `coef * 127 / max|coef|`, int() truncation.  weights[4][10] receives the new float table the playout
 * kernels read (intercept column 0), params[36] the stored integers ('A'.. order), fits[4][16] =
 * coef[9], intercept, rmse, r2, n, 0, 0, 0.  A shard without samples keeps its row of prev_weights.
 * All pointers DEVICE; weights may alias prev_weights. */
int othello_learn_solve(const double *stats, const float *prev_weights, float *weights, int32_t *params,
                        double *fits, void *stream);

/* One learning step's refit in ONE launch, straight from the (all-reduced) accumulators: othello_learn_stats +
 * othello_learn_solve, the statistics passing through shared memory (also written to `stats` if not NULL).
 * clear != 0 leaves acc zeroed for the next iteration's othello_learn_accumulate.  DEVICE pointers. */
int othello_learn_refit(int64_t *acc, int32_t clear, double *stats /* [4][112] or NULL */, const float *prev_weights,
                        float *weights, int32_t *params, double *fits, void *stream);

/* ---- the reference's value table, exactly ------------------------------------------------------ */

/* __update_state_for_a_book (progress_position_moves_learn.py:37-48): one (key, new_value) record per
 * (position, side) written AT ITS PLACE IN THE REFERENCE'S UPDATE ORDER -- games ascending, positions
 * terminal -> start (replearn.py:37-38), 'O' then 'X' (:44-47).  Game g's records start at rec_base[g]
 * (exclusive prefix sum of 2 * (nplies + 1), computed by the caller).  key = counts() packed into 43
 * bits: discs(7) mobility(6) a(3) b(4) c(3) d(4) e(4) f(5) g(3) h(4), most significant first. */
int othello_value_records(const uint64_t *traj_black, const uint64_t *traj_white, const int32_t *nplies,
                          const uint64_t *final_black, const uint64_t *final_white, int64_t n_games, int64_t stride,
                          int32_t t_max, const double *decay /* [t_max+1] */, const int64_t *rec_base,
                          uint64_t *keys, double *targets, void *stream);

/* Stable sort of n (key, value) records by the low `key_bits` bits of the key -- hand-written LSD radix
 * sort, 8 bits per pass, records of equal keys keep their order (= the reference's update order).  The
 * result is left in keys / values; *_alt are scratch of the same size.  workspace: DEVICE,
 * >= othello_sort_workspace_bytes(n).  n < 2^32. */
int64_t othello_sort_workspace_bytes(int64_t n);
int othello_sort_records(uint64_t *keys, double *values, uint64_t *keys_alt, double *values_alt, int64_t n,
                         int32_t key_bits, void *workspace, int64_t workspace_bytes, void *stream);

/* Stable partition of the records by the rank that owns their key when the table is sharded over `world`
 * GPUs (SURVEY 8e: one all_to_all of records per batch): out = records of owner 0, then owner 1, ...,
 * order preserved inside an owner; owner_counts[world] (DEVICE int64) receives the block sizes. */
int othello_partition_records(const uint64_t *keys, const double *values, uint64_t *keys_out, double *values_out,
                              int64_t n, int32_t world, int64_t *owner_counts, void *workspace, int64_t workspace_bytes,
                              void *stream);

/* The table: open-addressing hash (slot_keys[2^log2_capacity] uint64, 0 = empty; slot_idx int32) from key
 * to an index into the dense arrays dense_keys / dense_values.  __update_state_map (:50-62) for a SORTED
 * batch of records in two steps, so that the caller can grow the arrays in between:
 *   othello_table_probe: marks the heads of the runs of equal keys and looks them up; counters[1] (DEVICE
 *     int64[2]) = number of keys the batch adds.  workspace: DEVICE, >= othello_table_workspace_bytes(n),
 *     handed unchanged to othello_table_apply.
 *   othello_table_apply: new keys are appended to the dense arrays at n_before.. in key order, entered into
 *     the hash and start from 0 (`set(key, 0)`, :52-53); then every run is folded into its value in update
 *     order, V = new if V == 0 else V*(1-a) + new*a in fp64 with the reference's rounding (no fused
 *     multiply-add) -- short runs by one thread each, long runs (>= 128 records) by one warp each.  Needs
 *     2 * (n_before + new) <= 2^log2_capacity <= 2^30. */
int64_t othello_table_workspace_bytes(int64_t n);
int othello_table_probe(const uint64_t *sorted_keys, int64_t n, const uint64_t *slot_keys, const int32_t *slot_idx,
                        int32_t log2_capacity, void *workspace, int64_t workspace_bytes, int64_t *counters, void *stream);
int othello_table_apply(const uint64_t *sorted_keys, const double *sorted_targets, int64_t n, double a,
                        uint64_t *slot_keys, int32_t *slot_idx, int32_t log2_capacity, uint64_t *dense_keys,
                        double *dense_values, int64_t n_before, void *workspace, void *stream);
/* (re)build the hash from dense_keys[0..n) (slot arrays zeroed by the caller); key -> dense index or -1 */
int othello_table_rehash(const uint64_t *dense_keys, int64_t n, uint64_t *slot_keys, int32_t *slot_idx,
                         int32_t log2_capacity, void *stream);
int othello_table_lookup(const uint64_t *query, int64_t n, const uint64_t *slot_keys, const int32_t *slot_idx,
                         int32_t log2_capacity, int32_t *index, void *stream);

/* packed key -> the 10 integers of counts() (features[n][10]) */
int othello_unpack_keys(const uint64_t *keys, int32_t *features, int64_t n, void *stream);

/* ---- measurement helper --------------------------------------------------------------------- */

/* INT32 ALU-pipe micro-benchmark: every thread runs `iters` rounds of 8 independent LOP3/SHF
 * chains (32 integer lane-ops per round).  Used by bench.py to measure the integer roofline
 * denominator on the box.  sink: DEVICE uint32[blocks*threads]. */
int othello_int32_peak_kernel(uint32_t *sink, int blocks, int threads, int iters, void *stream);

/* Same, but every round is 16 LOP3 (ALU pipe) + 16 IMAD (FMA pipe): the integer ceiling of code that
 * spreads its work over both pipes (32 lane-ops per thread per round). */
int othello_int32_dual_peak_kernel(uint32_t *sink, int blocks, int threads, int iters, void *stream);

/* ---- host-buffer front end (what a non-torch caller binds) ----------------------------------- */

typedef struct othello_ctx othello_ctx;

int  othello_ctx_create(int device, othello_ctx **out);
void othello_ctx_destroy(othello_ctx *ctx);

/* The single-game facade (subproc_b200/board.py) in one call: Board.put(color, x, y) (board.py:161-174)
 * for move = x + 8*y in 0..63 -- the position is returned unchanged with ret = 0 when the square is
 * occupied or nothing flips -- or no move at all (move = OTHELLO_PASS or anything else), followed by what
 * the reference's callers ask about the resulting position before the next ply (game_runner.py:137,162,
 * 194-196; game_recorder.py:112; counts()): legal moves and counts() features of both colours, disc
 * counts.  One launch + one synchronise; the kernel writes `info` through mapped pinned memory. */
typedef struct {
    uint64_t black, white;        /* the position after the move */
    uint64_t flips;               /* discs flipped (0: put() returned 0) */
    uint64_t legal_black, legal_white;   /* Board.puttables(Black / White) as masks */
    int32_t  ret;                 /* Board.put's return value: number of discs flipped */
    int32_t  n_black, n_white, n_empty;
    int32_t  features_black[OTHELLO_FEATURES], features_white[OTHELLO_FEATURES];   /* counts(book, 'O' / 'X') */
} othello_position_info;
int othello_board_apply_host(othello_ctx *ctx, uint64_t black, uint64_t white, int32_t color, int32_t move,
                             othello_position_info *info);

/* puttables / put_s on host arrays: copies in, launches, copies out, synchronises. */
int othello_legal_host(othello_ctx *ctx, const uint64_t *own, const uint64_t *opp, uint64_t *legal, int64_t n);
int othello_step_host(othello_ctx *ctx, uint64_t *black, uint64_t *white, uint8_t *turn, int32_t *nturn,
                      const uint8_t *move, uint64_t *flips_out, int32_t *ret, uint8_t *flags, int64_t n);

/* tuning knobs of a context */
#define OTHELLO_OPT_MAX_CHUNKS 1   /* playout batches are pipelined in at most this many chunks (default 8) */
int othello_ctx_set_option(othello_ctx *ctx, int32_t option, int64_t value);

/* play_a_game for n games from host-resident start positions (NULL = standard opening); the
 * trajectory stays in device memory owned by the context (othello_ctx_trajectory) unless host
 * trajectory pointers are given.  Per-game results come back to the host arrays.  Synchronous:
 * othello_playout_host_async + othello_ctx_wait. */
int othello_playout_host(othello_ctx *ctx, uint64_t seed, uint64_t gid0, int64_t n_games,
                         const uint64_t *black0, const uint64_t *white0, const uint8_t *turn0,
                         int32_t policy, int32_t random_plies, int32_t n_rand_black, int32_t n_rand_white,
                         const float *weights /* host [4][10] or NULL */, int32_t policy_white /* -1 = same */,
                         const float *weights_white /* host [4][10] or NULL = same */, int32_t t_max,
                         uint64_t *traj_black, uint64_t *traj_white, uint8_t *traj_move /* host or NULL */,
                         int32_t *nplies, uint64_t *final_black, uint64_t *final_white);

/* The same, asynchronous: enqueues copy-in, kernels and copy-out and returns at once with a ticket;
 * the host output arrays (and `totals`: HOST int64[4], the sums of othello_playout_args.totals for
 * this batch, or NULL) are valid after othello_ctx_wait(ctx, ticket).  nplies / final_* / summary may each
 * be NULL: a caller that only needs who won and how long the games were takes `summary` (2 B per game
 * instead of 20), or just `totals`.  A context keeps two batches in
 * flight: issue batch i+1, then wait for batch i, and the PCIe copies of one batch run under the
 * kernels of the other.  Input arrays must stay untouched until the ticket has been waited for (use
 * pinned memory -- pageable buffers make the copies synchronous).  Issuing a third batch reuses the
 * device buffers of the first; if the caller has not waited for the first yet, the call does. */
int othello_playout_host_async(othello_ctx *ctx, uint64_t seed, uint64_t gid0, int64_t n_games,
                               const uint64_t *black0, const uint64_t *white0, const uint8_t *turn0,
                               int32_t policy, int32_t random_plies, int32_t n_rand_black, int32_t n_rand_white,
                               const float *weights, int32_t policy_white, const float *weights_white, int32_t t_max,
                               uint64_t *traj_black, uint64_t *traj_white, uint8_t *traj_move,
                               int32_t *nplies, uint64_t *final_black, uint64_t *final_white,
                               uint16_t *summary /* host [n], see othello_playout_args.summary, or NULL */,
                               int64_t *totals, int64_t *ticket);
int othello_ctx_wait(othello_ctx *ctx, int64_t ticket);

/* device pointers of the most recently ISSUED playout's trajectory ([t_max+1][n], [t_max+1][n],
 * [t_max][n]); valid once its ticket has been waited for and until two more playouts have been
 * issued on the context (or a *_legal_host / *_step_host call reuses the workspace) */
int othello_ctx_trajectory(othello_ctx *ctx, uint64_t **traj_black, uint64_t **traj_white, uint8_t **traj_move,
                           int64_t *stride, int32_t *t_max);

#ifdef __cplusplus
}
#endif
#endif /* OTHELLO_B200_H */
