/*
 * tests/solve_oracle.c -- TEST INFRASTRUCTURE: exact endgame values on the
 * oracle's mailbox rules, the reference the solver (othello_solve) is checked
 * against.  It includes oracle/othello_oracle.c as it stands, so it shares the
 * oracle's rules (puttables, put_move, is_game_over -- board.py) and no code
 * with the bitboard search it checks.
 *
 * value = own - opponent discs of the terminal position under perfect play,
 * own = the side to move; the game ends when neither side can move
 * (board.py:57-58), a pass is a ply, and empty squares left at the end are not
 * given to the winner (winner by disc count, game_runner.py:194-199; target
 * own - opp final discs, progress_position_moves_learn.py:55).  move = lowest
 * square reaching the value, 64 = must pass, 255 = game over; a position with
 * more than 24 empties or overlapping colours: value -128, move 255.
 */
#include "../oracle/othello_oracle.c"

static int disc_diff(const board_t *b)
{
    return count_cells(b, b->turn) - count_cells(b, hostile(b->turn));
}

/* plain negamax, no pruning; children in ascending square order */
static int minimax(const board_t *b)
{
    uint64_t moves = puttables(b, b->turn);
    if (moves == 0) {
        if (n_puttable_for(b, hostile(b->turn)) == 0) return disc_diff(b);
        board_t c = *b; put_move(&c, 64, 0);
        return -minimax(&c);
    }
    int best = -65;
    for (int s = 0; s < 64; s++) if ((moves >> s) & 1) {
        board_t c = *b; put_move(&c, s, 0);
        int v = -minimax(&c);
        if (v > best) best = v;
    }
    return best;
}

/* plain fail-hard alpha-beta, no move ordering: exact when the value lies
 * strictly inside (alpha, beta); otherwise at most alpha / at least beta */
static int alphabeta(const board_t *b, int alpha, int beta)
{
    uint64_t moves = puttables(b, b->turn);
    if (moves == 0) {
        if (n_puttable_for(b, hostile(b->turn)) == 0) return disc_diff(b);
        board_t c = *b; put_move(&c, 64, 0);
        return -alphabeta(&c, -beta, -alpha);
    }
    for (int s = 0; s < 64; s++) if ((moves >> s) & 1) {
        board_t c = *b; put_move(&c, s, 0);
        int v = -alphabeta(&c, -beta, -alpha);
        if (v >= beta) return beta;
        if (v > alpha) alpha = v;
    }
    return alpha;
}

/* the root: children in ascending square order, a strict > keeps the lowest
 * square.  With pruning, the window (best, 65) makes a child's value exact
 * exactly when it beats the best so far. */
static int solve_root(uint64_t black, uint64_t white, int turn, int pruned, int *move)
{
    board_t b; cells_from_bits(&b, black, white); b.turn = turn; b.nturn = 0;
    *move = 255;
    if ((black & white) || count_cells(&b, EMPTY) > 24) return -128;
    uint64_t moves = puttables(&b, b.turn);
    if (moves == 0) {
        if (n_puttable_for(&b, hostile(b.turn)) == 0) return disc_diff(&b);
        board_t c = b; put_move(&c, 64, 0);
        *move = 64;
        return -(pruned ? alphabeta(&c, -65, 65) : minimax(&c));
    }
    int best = -65;
    for (int s = 0; s < 64; s++) if ((moves >> s) & 1) {
        board_t c = b; put_move(&c, s, 0);
        int v = -(pruned ? alphabeta(&c, -65, -best) : minimax(&c));
        if (v > best) { best = v; *move = s; }
    }
    return best;
}

int orc_solve_minimax(uint64_t black, uint64_t white, int turn, int *move)
{
    return solve_root(black, white, turn, 0, move);
}

int orc_solve_ab(uint64_t black, uint64_t white, int turn, int *move)
{
    return solve_root(black, white, turn, 1, move);
}

/* pruned = 0: orc_solve_minimax, 1: orc_solve_ab; turn 1 = Black, anything else = White */
void orc_solve_batch(const uint64_t *black, const uint64_t *white, const uint8_t *turn, int pruned,
                     int32_t *value, uint8_t *move, int64_t n)
{
    for (int64_t i = 0; i < n; i++) {
        int m;
        value[i] = solve_root(black[i], white[i], turn[i] == BLACK ? BLACK : WHITE, pruned, &m);
        move[i] = (uint8_t)m;
    }
}
