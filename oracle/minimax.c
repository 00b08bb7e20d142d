/* TEST INFRASTRUCTURE ONLY -- C restatement of oracle/minimax_ref.py (the reference's depth-limited OptimalPlayer,
 * src/reversi/players/reversi_players.py:35-77): plain minimax, NO pruning, so it checks the GPU kernel's alpha-beta
 * independently.  Rules: one direction at a time on bitboards (bit = row*8 + col), and a ray walk for the flips, written
 * apart from the fills of betazero_b200/csrc/bitboard.cuh.  Built by oracle/pyminimax.py. */
#include <stdint.h>

#define INF 127

static const int DR[8] = {-1, -1, -1, 0, 0, 1, 1, 1};
static const int DC[8] = {-1, 0, 1, -1, 1, -1, 0, 1};

/* discs flipped by `mover` placing on (r, c); 0 when the move is not valid (reversi_board.py:25-59) */
static uint64_t flips(uint64_t me, uint64_t opp, int size, int r, int c) {
    if (((me | opp) >> (r * 8 + c)) & 1) return 0;
    uint64_t all = 0;
    for (int d = 0; d < 8; ++d) {
        uint64_t run = 0;
        int rr = r + DR[d], cc = c + DC[d];
        while (rr >= 0 && rr < size && cc >= 0 && cc < size && ((opp >> (rr * 8 + cc)) & 1)) {
            run |= 1ull << (rr * 8 + cc);
            rr += DR[d];
            cc += DC[d];
        }
        if (run && rr >= 0 && rr < size && cc >= 0 && cc < size && ((me >> (rr * 8 + cc)) & 1)) all |= run;
    }
    return all;
}

/* one step of every disc in direction d, discs that would wrap around a row dropped */
static uint64_t step(uint64_t b, int d) {
    const uint64_t not_a = 0xFEFEFEFEFEFEFEFEull, not_h = 0x7F7F7F7F7F7F7F7Full;
    const int s = DR[d] * 8 + DC[d];
    b = s > 0 ? b << s : b >> -s;
    return DC[d] > 0 ? b & not_a : (DC[d] < 0 ? b & not_h : b);
}

/* generate_possible_moves as a mask: one direction at a time, a run of opponent discs grown one step per pass */
static uint64_t moves_of(uint64_t me, uint64_t opp, int size) {
    uint64_t cells = 0;
    for (int r = 0; r < size; ++r)
        for (int c = 0; c < size; ++c) cells |= 1ull << (r * 8 + c);
    const uint64_t empty = ~(me | opp) & cells;
    uint64_t m = 0;
    for (int d = 0; d < 8; ++d) {
        uint64_t t = step(me, d) & opp;
        for (int k = 0; k < 5; ++k) t |= step(t, d) & opp;
        m |= step(t, d) & empty;
    }
    return m;
}

/* node (me, opp) with `me` to move at `depth`; the player is `me` at even depths */
static int minimax(uint64_t me, uint64_t opp, int size, int depth, int max_depth, int64_t *nodes) {
    ++*nodes;
    const int maxing = (depth & 1) == 0;
    const int ev = maxing ? __builtin_popcountll(me) - __builtin_popcountll(opp)
                          : __builtin_popcountll(opp) - __builtin_popcountll(me);
    if (depth >= max_depth) return ev;
    const uint64_t m = moves_of(me, opp, size);
    if (m == 0 && moves_of(opp, me, size) == 0) return ev;
    int best = maxing ? -INF : INF;
    for (int a = 0; a < 64; ++a) {
        if (!((m >> a) & 1)) continue;
        const uint64_t x = 1ull << a, f = flips(me, opp, size, a >> 3, a & 7);
        const int v = minimax(opp & ~f, me | x | f, size, depth + 1, max_depth, nodes);
        if (maxing ? v > best : v < best) best = v;
    }
    return best;
}

static uint32_t philox_u32(uint64_t seed, uint64_t key, uint32_t counter) {
    uint32_t c0 = (uint32_t)key, c1 = (uint32_t)(key >> 32), c2 = counter, c3 = 0;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c0;
}

/* the search of bz_minimax_moves for every root (include/betazero_b200.h); OpenMP over roots */
void orc_minimax_moves(const uint64_t *me, const uint64_t *opp, const uint8_t *depth, const uint64_t *key, uint64_t seed,
                       int64_t n, int size, uint8_t *action, int8_t *value, int64_t *nodes) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t i = 0; i < n; ++i) {
        const uint64_t M = me[i], O = opp[i];
        const int D = depth[i];
        int64_t nd = 1;
        const uint64_t m = moves_of(M, O, size);
        const int ev = __builtin_popcountll(M) - __builtin_popcountll(O);
        int act = -1, val;
        if (m == 0) {
            const int over = moves_of(O, M, size) == 0;
            act = over ? 255 : 64;
            val = (D == 0 || over) ? ev : -INF;
        } else if (D == 0) {
            val = ev;
        } else {
            val = -INF;
            for (int a = 0; a < 64; ++a) {
                if (!((m >> a) & 1)) continue;
                const uint64_t x = 1ull << a, f = flips(M, O, size, a >> 3, a & 7);
                const int v = minimax(O & ~f, M | x | f, size, 1, D, &nd);
                if (v > val) {
                    val = v;
                    act = a;
                }
            }
        }
        if (act < 0) { /* no move from the search: the Philox move */
            const uint32_t u = philox_u32(seed, (1ull << 32) + key[i], (uint32_t)__builtin_popcountll(M | O));
            int k = (int)(((uint64_t)u * (uint64_t)__builtin_popcountll(m)) >> 32);
            for (int a = 0; a < 64; ++a) {
                if (!((m >> a) & 1)) continue;
                if (k-- == 0) {
                    act = a;
                    break;
                }
            }
        }
        action[i] = (uint8_t)act;
        value[i] = (int8_t)val;
        nodes[i] = nd;
    }
}
