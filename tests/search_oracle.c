/*
 * tests/search_oracle.c -- TEST INFRASTRUCTURE: depth-limited minimax values
 * on the oracle's mailbox rules and its fp64 evaluation, the reference the
 * midgame search (othello_search) is checked against.  It includes
 * oracle/othello_oracle.c as it stands, so it shares the oracle's rules
 * (puttables, put_move, is_game_over -- board.py) and evaluation and no code
 * with the bitboard search it checks.
 *
 * Every node is scored from the root mover's side: evaluate(node, root, w).
 * A pass is a ply and uses one level of depth; a node is a leaf `depth` plies
 * below the root or when neither side can move.  Max on the root mover's
 * plies, min on the opponent's.  move = lowest square reaching the value,
 * 64 = the root mover must pass (value: the passed position to depth - 1),
 * 255 = game over (value: the root's score); overlapping colours: NaN, 255.
 * With integer weights every score is an integer, exact in fp32 and fp64.
 */
#include "../oracle/othello_oracle.c"

/* plain minimax, no pruning; children in ascending square order */
static double minimax(const board_t *b, int root, int depth, const double *w)
{
    if (depth == 0 || is_game_over(b)) return evaluate(b, root, w);
    uint64_t moves = puttables(b, b->turn);
    if (moves == 0) {
        board_t c = *b; put_move(&c, 64, 0);
        return minimax(&c, root, depth - 1, w);
    }
    int maxing = b->turn == root;
    double best = maxing ? -INFINITY : INFINITY;
    for (int s = 0; s < 64; s++) if ((moves >> s) & 1) {
        board_t c = *b; put_move(&c, s, 0);
        double v = minimax(&c, root, depth - 1, w);
        if (maxing ? v > best : v < best) best = v;
    }
    return best;
}

/* plain fail-hard alpha-beta, no move ordering: exact when the value lies
 * strictly inside (alpha, beta); otherwise at most alpha / at least beta */
static double alphabeta(const board_t *b, int root, int depth, double alpha, double beta, const double *w)
{
    if (depth == 0 || is_game_over(b)) return evaluate(b, root, w);
    uint64_t moves = puttables(b, b->turn);
    if (moves == 0) {
        board_t c = *b; put_move(&c, 64, 0);
        return alphabeta(&c, root, depth - 1, alpha, beta, w);
    }
    int maxing = b->turn == root;
    for (int s = 0; s < 64; s++) if ((moves >> s) & 1) {
        board_t c = *b; put_move(&c, s, 0);
        double v = alphabeta(&c, root, depth - 1, alpha, beta, w);
        if (maxing) {
            if (v >= beta) return beta;
            if (v > alpha) alpha = v;
        } else {
            if (v <= alpha) return alpha;
            if (v < beta) beta = v;
        }
    }
    return maxing ? alpha : beta;
}

/* the root: children in ascending square order, a strict > keeps the lowest
 * square.  With pruning, the window (best, +inf) makes a child's value exact
 * exactly when it beats the best so far. */
static double search_root(uint64_t black, uint64_t white, int turn, const double *w, int depth, int pruned, int *move)
{
    board_t b; cells_from_bits(&b, black, white); b.turn = turn; b.nturn = 0;
    *move = 255;
    if (black & white) return NAN;
    if (is_game_over(&b)) return evaluate(&b, turn, w);
    uint64_t moves = puttables(&b, turn);
    if (moves == 0) {
        board_t c = b; put_move(&c, 64, 0);
        *move = 64;
        return pruned ? alphabeta(&c, turn, depth - 1, -INFINITY, INFINITY, w) : minimax(&c, turn, depth - 1, w);
    }
    double best = -INFINITY;
    for (int s = 0; s < 64; s++) if ((moves >> s) & 1) {
        board_t c = b; put_move(&c, s, 0);
        double v = pruned ? alphabeta(&c, turn, depth - 1, *move == 255 ? -INFINITY : best, INFINITY, w)
                          : minimax(&c, turn, depth - 1, w);
        if (*move == 255 || v > best) { best = v; *move = s; }
    }
    return best;
}

/* the minimax value of every root move's subtree, from the root mover's side (NaN where the move is not legal) */
void orc_search_children(uint64_t black, uint64_t white, int turn, const double *w, int depth, double out[64])
{
    board_t b; cells_from_bits(&b, black, white); b.turn = turn == BLACK ? BLACK : WHITE; b.nturn = 0;
    uint64_t moves = puttables(&b, b.turn);
    for (int s = 0; s < 64; s++) {
        out[s] = NAN;
        if ((moves >> s) & 1) { board_t c = b; put_move(&c, s, 0); out[s] = minimax(&c, b.turn, depth - 1, w); }
    }
}

/* w: [4][10]; pruned = 0: plain minimax, 1: unordered alpha-beta; turn 1 = Black, anything else = White */
void orc_search_batch(const uint64_t *black, const uint64_t *white, const uint8_t *turn, const double *w, int depth,
                      int pruned, double *value, uint8_t *move, int64_t n)
{
    for (int64_t i = 0; i < n; i++) {
        int m;
        value[i] = search_root(black[i], white[i], turn[i] == BLACK ? BLACK : WHITE, w, depth, pruned, &m);
        move[i] = (uint8_t)m;
    }
}
