/* TEST INFRASTRUCTURE ONLY -- C restatement of oracle/endgame_ref.py (the exact endgame value of bz_endgame_solve):
 * plain negamax to the end of the game, NO pruning, so it checks the GPU kernel's alpha-beta independently.  The rules
 * are minimax.c's (moves_of, flips: one direction at a time and a ray walk, written apart from
 * betazero_b200/csrc/bitboard.cuh), included here rather than copied.  Built by oracle/pyendgame.py. */
#include "minimax.c"

/* the value of (me, opp), `me` to move; a pass is entered as the position with the sides swapped; every position
 * entered counts one node */
static int negamax(uint64_t me, uint64_t opp, int size, int64_t *nodes) {
    ++*nodes;
    const uint64_t m = moves_of(me, opp, size);
    if (m == 0) {
        if (moves_of(opp, me, size) == 0) return __builtin_popcountll(me) - __builtin_popcountll(opp);
        return -negamax(opp, me, size, nodes);
    }
    int best = -128;
    for (int a = 0; a < 64; ++a) {
        if (!((m >> a) & 1)) continue;
        const uint64_t x = 1ull << a, f = flips(me, opp, size, a >> 3, a & 7);
        const int v = -negamax(opp & ~f, me | x | f, size, nodes);
        if (v > best) best = v;
    }
    return best;
}

/* the results of bz_endgame_solve for every root; OpenMP over roots.  move_value: [n * 65] */
void orc_endgame_solve(const uint64_t *me, const uint64_t *opp, int64_t n, int size, uint8_t *action, int8_t *value,
                       int8_t *move_value, int64_t *nodes) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t i = 0; i < n; ++i) {
        const uint64_t M = me[i], O = opp[i];
        int8_t *mv = move_value + i * 65;
        for (int a = 0; a < 65; ++a) mv[a] = -128;
        int64_t nd = 1;
        const uint64_t m = moves_of(M, O, size);
        int act = 255, val;
        if (m == 0 && moves_of(O, M, size) == 0) {
            val = __builtin_popcountll(M) - __builtin_popcountll(O);
        } else if (m == 0) {
            val = mv[64] = (int8_t)-negamax(O, M, size, &nd);
            act = 64;
        } else {
            val = -128;
            for (int a = 0; a < 64; ++a) {
                if (!((m >> a) & 1)) continue;
                const uint64_t x = 1ull << a, f = flips(M, O, size, a >> 3, a & 7);
                const int v = -negamax(O & ~f, M | x | f, size, &nd);
                mv[a] = (int8_t)v;
                if (v > val) {
                    val = v;
                    act = a;
                }
            }
        }
        action[i] = (uint8_t)act;
        value[i] = (int8_t)val;
        nodes[i] = nd;
    }
}
