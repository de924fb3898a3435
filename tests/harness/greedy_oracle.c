/*
 * greedy_oracle.c -- CPU restatement of the greedy agent.   TEST INFRASTRUCTURE ONLY.
 *
 * The greedy agent has no counterpart in the reference, so its restatement is kept apart from oracle/azul_oracle.c (the
 * file the golden traces pin to the reference) and is compiled together with it: it uses the oracle's own unpacked rule
 * functions, and it is written the naive way -- copy the game, move, score, for every legal action -- so that it is an
 * independent statement of the spec the kernels implement with per-(line, colour) arithmetic.
 */
#include "../../oracle/azul_oracle.c"

/* SPEC of the greedy agent (shared with greedy_action in csrc/azb_rules.cuh):
 *   v(a) = the mover's score after Azul.move(a) (azul.py:118-161) and count_score (azul.py:192-295) on a copy, WITHOUT
 *          the clamp at zero of azul.py:294-295: score + count_floor + count_wall of the mover.
 *   T    = the legal actions of largest v, in ascending action index (a = d + 6c + 30p).
 *   pick = T[mulhi(word, |T|)], word = the random agent's word of this env step (word total_steps & 3 of
 *          Philox(gid, total_steps >> 2, ACTION, 0)); -1 when no action is legal. */
static int greedy_action(const ao_game *g, int pool, uint32_t word)
{
    int best = 0, n_best = 0, T[180];
    for (int a = 0; a < 180; a++) {
        int d = a % 6, c = (a / 6) % 5, p = a / 30;
        if (!is_legal_move(g, d, c, p)) continue;
        ao_game cp = *g;
        int s = seat(&cp);
        move(&cp, pool, d, c, p);
        int v = cp.score[s] + count_floor(&cp, s) + count_wall(&cp, pool, s);
        if (n_best == 0 || v > best) { best = v; n_best = 0; }
        if (v == best) T[n_best++] = a;
    }
    if (n_best == 0) return -1;
    return T[mulhi32(word, (uint32_t)n_best)];
}

int ao_greedy_action(const int32_t *rec, int players, int pool, uint32_t word)
{
    ao_game g; from_record(&g, rec, players);
    return greedy_action(&g, pool, word);
}

/* the number of legal actions that share the largest v (test statistics: states with ties) */
int ao_greedy_ties(const int32_t *rec, int players, int pool)
{
    ao_game g; from_record(&g, rec, players);
    int best = 0, n_best = 0;
    for (int a = 0; a < 180; a++) {
        int d = a % 6, c = (a / 6) % 5, p = a / 30;
        if (!is_legal_move(&g, d, c, p)) continue;
        ao_game cp = g;
        int s = seat(&cp);
        move(&cp, pool, d, c, p);
        int v = cp.score[s] + count_floor(&cp, s) + count_wall(&cp, pool, s);
        if (n_best == 0 || v > best) { best = v; n_best = 0; }
        if (v == best) n_best++;
    }
    return n_best;
}

/* SPEC of azb_opponent_greedy: ao_opponent_random's loop and return value with the greedy agent's pick */
int ao_opponent_greedy(int32_t *rec, int players, int pool, uint64_t seed, uint32_t gid, int require_two, uint32_t *mask6)
{
    ao_game g; from_record(&g, rec, players);
    for (;;) {
        legal_mask(&g, mask6);
        if (g.end_of_game) break;                                        /* game_runner.py:46 */
        int n_valid = 0;
        for (int p = 0; p < 6; p++) n_valid += __builtin_popcount(mask6[p]);
        if (g.current_player == 1 && (!require_two || n_valid >= 2)) break;
        if (n_valid == 0) { g.status |= ST_STUCK; break; }
        uint32_t w[4];
        draw_words(seed, gid, g.total_steps >> 2, PURPOSE_ACTION, 0, w);
        int a = greedy_action(&g, pool, w[g.total_steps & 3]);
        step(&g, pool, a % 6, (a / 6) % 5, a / 30, NULL, seed, gid);
    }
    to_record(&g, rec, players);
    ao_game cp = g;                                                      /* game_runner.py:48-50 */
    count_score(&cp, pool);
    return cp.score[0] - cp.score[1];
}
