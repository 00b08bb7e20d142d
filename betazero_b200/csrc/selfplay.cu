// Lockstep self-play driver kernels for sm_100a: the batched form of the reference episode loop
// (src/reversi/game_logic/reversi_terminal.py:16-38): after a search, every game slot picks its
// move from the root visit counts, records (board, pi), applies the move (or pass), tests for the
// end of the game (reversi_board.py:61-65), scores finished games (get_score, :67-76), flushes
// them to the replay buffer and restarts the slot.  One warp per game slot == per tree.
#include "bitboard.cuh"
#include "common.cuh"

namespace bz {
namespace {

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kWarpsPerCta = 4;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int A = BZ_REVERSI_ACTIONS;

// ---- Philox4x32-10 (counter-based RNG; results depend only on (seed, game id, ply)) -------------
__host__ __device__ inline uint32_t philox_u32(uint64_t seed, uint64_t game_id, uint32_t ply) {
    uint32_t c0 = (uint32_t)game_id, c1 = (uint32_t)(game_id >> 32), c2 = ply, c3 = 0;
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

__global__ void __launch_bounds__(256) selfplay_init_kernel(const bz_selfplay_state S, int64_t first_game_id) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < 8) S.counters[s] = 0ull;
    if (s >= S.n_games) return;
    S.me[s] = start_me(S.board_size);
    S.opp[s] = start_opp(S.board_size);
    S.player[s] = 1;
    S.ply[s] = 0;
    S.game_id[s] = first_game_id + s;
}

__global__ void __launch_bounds__(kThreads)
    selfplay_advance_kernel(const bz_selfplay_state S, const bz_tree_pools P, uint8_t *action_out, uint64_t cells) {
    const int s = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (s >= S.n_games) return;
    const int lane = threadIdx.x & 31;

    // root statistics: lane i holds edge i (ascending action id); a 33rd edge is read uniformly
    const uint32_t rmeta = P.root_meta[s];
    const int n = (int)((rmeta >> BZ_META_N_SHIFT) & 63u);
    const uint32_t *blk = P.arena + (int64_t)s * P.arena_units * 8 + (int64_t)(rmeta >> BZ_META_OFF_SHIFT) * 8;
    int Ne = 0, N32 = 0;
    unsigned act = 127u, act32 = 127u;
    if (lane < n) {
        Ne = (int)blk[BZ_NODE_HEADER_WORDS + lane];
        act = blk[BZ_NODE_HEADER_WORDS + 3 * n + lane] & 127u;
    }
    if (n > 32) {
        N32 = (int)blk[BZ_NODE_HEADER_WORDS + 32];
        act32 = blk[BZ_NODE_HEADER_WORDS + 3 * n + 32] & 127u;
    }
    const int total = __reduce_add_sync(kFull, Ne) + N32;
    const int ply = S.ply[s];
    const int64_t gid = S.game_id[s];
    uint64_t me = S.me[s], opp = S.opp[s];
    const int player = S.player[s];

    // --- choose the move -------------------------------------------------------------------
    unsigned action;
    if (n == 0 || total == 0) {
        // no search result (cannot happen for a live game searched with >= 2 iterations): fall back
        // to the first legal move so the game still advances deterministically
        const uint64_t m = legal_mask(me, opp, cells);
        action = m ? (unsigned)(__ffsll((long long)m) - 1) : 64u;
    } else if (ply < S.temp_plies) {
        // sample ~ N: first edge whose inclusive prefix sum exceeds floor(u32 * total / 2^32)
        const uint32_t r = philox_u32(S.seed, (uint64_t)gid, (uint32_t)ply);
        const int target = (int)(((uint64_t)r * (uint64_t)total) >> 32);
        int cum = Ne;
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(kFull, cum, d);
            if (lane >= d) cum += up;
        }
        const unsigned hit = __ballot_sync(kFull, lane < n && cum > target);
        action = hit ? __shfl_sync(kFull, act, __ffs(hit) - 1) : act32;
    } else {
        // most visited, lowest action id on ties (players.py:92-98 applied to visit counts)
        unsigned key = (lane < n && Ne > 0) ? (((unsigned)Ne << 7) | (127u - act)) : 0u;
        if (n > 32 && N32 > 0) {
            const unsigned k32 = ((unsigned)N32 << 7) | (127u - act32);
            key = k32 > key ? k32 : key;
        }
        key = __reduce_max_sync(kFull, key);
        action = 127u - (key & 127u);
    }

    // --- record (board, pi, player, action) in the slot's history -----------------------------
    const int64_t h = (int64_t)s * S.max_plies + ply;
    BZ_CHECK(s >= 0 && s < S.n_games && ply >= 0 && ply < S.max_plies && action <= 64u, 21);  // history row, move
    float *pi = S.hist_pi + h * A;
    for (int a = lane; a < A; a += 32) pi[a] = 0.f;
    __syncwarp();
    const float ftot = (float)(total > 0 ? total : 1);
    if (lane < n) pi[act] = __fdiv_rn((float)Ne, ftot);
    if (n > 32 && lane == 0) pi[act32] = __fdiv_rn((float)N32, ftot);
    if (total == 0 && lane == 0) pi[action] = 1.0f;
    if (lane == 0) {
        S.hist_me[h] = me;
        S.hist_opp[h] = opp;
        S.hist_player[h] = (int8_t)player;
        S.hist_action[h] = (uint8_t)action;
        if (action_out) action_out[s] = (uint8_t)action;
    }

    // --- apply, terminal test -----------------------------------------------------------------
    apply_legal(me, opp, action);  // now the NEXT mover's view; next player = -player
    const bool over = (legal_mask(me, opp, cells) | legal_mask(opp, me, cells)) == 0;
    const int nrec = ply + 1;
    if (!over && nrec < S.max_plies) {
        if (lane == 0) {
            S.me[s] = me;
            S.opp[s] = opp;
            S.player[s] = (int8_t)(-player);
            S.ply[s] = nrec;
            atomicAdd(&S.counters[1], 1ull);
        }
        return;
    }

    // --- finished: score, flush the history to the replay buffer, restart the slot ----------------
    const int cm = __popcll(me), co = __popcll(opp);
    const int winner = ((cm > co) - (cm < co)) * (-player);  // absolute: +1 X, -1 O, 0 draw
    // counters[0] = rows COMMITTED to the replay buffer: a game reserves its rows with a compare-and-swap and takes
    // nothing when it does not fit, so [0, counters[0]) never contains a row that no game wrote
    unsigned long long rb = ~0ull;  // ~0: no room, the game is dropped (counted in counters[5])
    if (lane == 0) {
        unsigned long long cur = S.counters[0];
        while (cur + (unsigned long long)nrec <= (unsigned long long)S.replay_cap) {
            const unsigned long long seen = atomicCAS(&S.counters[0], cur, cur + (unsigned long long)nrec);
            if (seen == cur) {
                rb = cur;
                break;
            }
            cur = seen;
        }
        atomicAdd(&S.counters[1], 1ull);
        atomicAdd(&S.counters[3 + winner], 1ull);
        atomicAdd(&S.counters[6], 1ull);
    }
    rb = __shfl_sync(kFull, rb, 0);
    __syncwarp();  // the record written above is visible to the copying lanes
    const int64_t h0 = (int64_t)s * S.max_plies;
    if (rb != ~0ull) {
        BZ_CHECK(rb + (unsigned long long)nrec <= (unsigned long long)S.replay_cap && nrec <= S.max_plies, 22);  // replay rows
        for (int r = lane; r < nrec; r += 32) {
            S.rp_me[rb + r] = S.hist_me[h0 + r];
            S.rp_opp[rb + r] = S.hist_opp[h0 + r];
            S.rp_z[rb + r] = (int8_t)(winner * S.hist_player[h0 + r]);
            S.rp_game[rb + r] = gid;
            S.rp_ply[rb + r] = (int16_t)r;
        }
        const int64_t nf = (int64_t)nrec * A;  // pi rows are contiguous in both buffers
        const float *src = S.hist_pi + h0 * A;
        float *dst = S.rp_pi + (int64_t)rb * A;
        for (int64_t i = lane; i < nf; i += 32) dst[i] = src[i];
    } else if (lane == 0) {
        atomicAdd(&S.counters[5], (unsigned long long)nrec);
    }
    if (lane == 0) {
        S.me[s] = start_me(S.board_size);
        S.opp[s] = start_opp(S.board_size);
        S.player[s] = 1;
        S.ply[s] = 0;
        S.game_id[s] = gid + S.id_stride;
    }
}

__global__ void __launch_bounds__(256)
    philox_kernel(uint64_t seed, const int64_t *game_id, const int32_t *ply, uint32_t *out, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = philox_u32(seed, (uint64_t)game_id[i], (uint32_t)ply[i]);
}


// ---- replay augmentation: dihedral transforms of (board, pi) records --------------------------------
// destination cell of source cell (r, c) on an n x n board under transform k (train.py:27-36)
__host__ __device__ inline int sym_cell(int k, int r, int c, int n) {
    const int m = n - 1;
    int nr, nc;
    switch (k) {
        case 1: nr = m - r; nc = c; break;      // flip(dims=[0])
        case 2: nr = r; nc = m - c; break;      // flip(dims=[1])
        case 3: nr = m - c; nc = r; break;      // rot90 x1: new[i][j] = old[j][m-i]
        case 4: nr = m - r; nc = m - c; break;  // rot90 x2
        case 5: nr = c; nc = m - r; break;      // rot90 x3: new[i][j] = old[m-j][i]
        case 6: nr = c; nc = r; break;          // transpose
        case 7: nr = m - c; nc = m - r; break;  // anti-transpose
        default: nr = r; nc = c; break;
    }
    return nr * 8 + nc;
}

__global__ void __launch_bounds__(256)
    symmetry_kernel(const uint64_t *__restrict__ me, const uint64_t *__restrict__ opp, const float *__restrict__ pi,
                    const uint8_t *__restrict__ sym, uint64_t *__restrict__ me_out, uint64_t *__restrict__ opp_out,
                    float *__restrict__ pi_out, int64_t n, int size) {
    const int64_t total = n * A;
    for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = g / A;
        const int a = (int)(g - i * A);
        const int k = sym[i] & 7;
        if (a == 64) {
            pi_out[g] = pi[g];  // pass is invariant; this thread also transforms the two bitboards
            uint64_t m = 0, o = 0;
            for (uint64_t b = me[i]; b; b &= b - 1) {
                const int s = __ffsll((long long)b) - 1;
                m |= 1ull << sym_cell(k, s >> 3, s & 7, size);
            }
            for (uint64_t b = opp[i]; b; b &= b - 1) {
                const int s = __ffsll((long long)b) - 1;
                o |= 1ull << sym_cell(k, s >> 3, s & 7, size);
            }
            me_out[i] = m;
            opp_out[i] = o;
        } else {
            const int r = a >> 3, c = a & 7;
            if (r < size && c < size) pi_out[i * A + sym_cell(k, r, c, size)] = pi[g];
            else pi_out[g] = 0.f;  // cells outside the board keep their (zero) slot
        }
    }
}

// 64-bit content hash of a (board, pi) record: the dedup key of the dataset expansion (a warp per record)
__device__ __forceinline__ uint64_t rec_mix(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__global__ void __launch_bounds__(256)
    record_hash_kernel(const uint64_t *__restrict__ me, const uint64_t *__restrict__ opp, const float *__restrict__ pi,
                       uint64_t *__restrict__ out, int64_t n) {
    const int lane = threadIdx.x & 31;
    for (int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; i < n; i += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const float *row = pi + i * A;
        uint64_t h = 0;
        for (int a = lane; a < A; a += 32) {
            const float f = row[a];
            const uint32_t bits = f == 0.f ? 0u : __float_as_uint(f);  // -0 == +0, as in a value comparison
            h += rec_mix(((uint64_t)(a + 1) << 32) | bits);           // order-independent sum of per-cell hashes
        }
        for (int d = 16; d; d >>= 1) h += __shfl_xor_sync(kFull, h, d);
        if (lane == 0) out[i] = rec_mix(h ^ rec_mix(me[i] + 0x9E3779B97F4A7C15ULL) ^ rec_mix(opp[i] * 0xD1B54A32D192ED03ULL + 1));
    }
}

// ---- net-versus-net matches ------------------------------------------------------------------------------------------
// Games 2i and 2i+1 are pair i: same opening, then net A (the pair's first entrant) is X in game 2i and O in game 2i+1.
constexpr int kPairTrees = BZ_MATCH_TREES_PER_PAIR;
constexpr int kLayoutThreads = 1024;

// the game has ended with (me, opp) seen by `player` to move: result (get_score: more discs wins), counts, counters
__device__ void match_finish(const bz_match_state &S, int g, uint64_t me, uint64_t opp, int player) {
    const int cx = __popcll(player > 0 ? me : opp), co = __popcll(player > 0 ? opp : me);
    const int winner = (cx > co) - (cx < co);  // absolute: +1 X, -1 O, 0 draw
    BZ_CHECK(g >= 0 && g < S.n_games, 30);  // game row
    S.result[g] = (int8_t)winner;
    S.count_x[g] = (uint8_t)cx;
    S.count_o[g] = (uint8_t)co;
    const int a_colour = (g & 1) ? -1 : 1;  // net A is X in even games
    const int r = winner * a_colour;
    unsigned long long *c = reinterpret_cast<unsigned long long *>(S.counters);
    atomicAdd(&c[3], 1ull);
    atomicAdd(&c[r > 0 ? 4 : (r == 0 ? 5 : 6)], 1ull);
    atomicAdd(&c[7], (unsigned long long)(long long)((cx - co) * a_colour));  // two's complement: signed sum
}

__device__ __forceinline__ bool game_over(uint64_t me, uint64_t opp, uint64_t cells) {
    return (legal_mask(me, opp, cells) | legal_mask(opp, me, cells)) == 0;
}

// a thread per game: start position, the pair's random opening, scoring of games that end inside it
__global__ void __launch_bounds__(256) match_init_kernel(const bz_match_state S, uint64_t cells) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= S.n_games) return;
    uint64_t me = start_me(S.board_size), opp = start_opp(S.board_size);
    int player = 1, ply = 0;
    uint8_t *mv = S.moves + (int64_t)g * BZ_MATCH_MAX_PLIES;
    for (int k = 0; k < BZ_MATCH_MAX_PLIES; ++k) mv[k] = 255u;
    const uint64_t pair_id = (uint64_t)(S.first_pair_id + g / 2);
    bool over = game_over(me, opp, cells);
    while (!over && ply < S.opening_plies && ply < BZ_MATCH_MAX_PLIES) {
        const uint64_t m = legal_mask(me, opp, cells);
        unsigned action = 64u;  // pass: the mover has no move (the game is not over, so the opponent has one)
        if (m) {
            // the k-th legal move in ascending cell order, k = floor(u32 * moves / 2^32)
            const uint32_t r = philox_u32(S.seed, pair_id, (uint32_t)ply);
            int k = (int)(((uint64_t)r * (uint64_t)__popcll(m)) >> 32);
            uint64_t b = m;
            for (; k > 0; --k) b &= b - 1;
            action = (unsigned)(__ffsll((long long)b) - 1);
        }
        BZ_CHECK(ply >= 0 && ply < BZ_MATCH_MAX_PLIES, 31);  // move row
        mv[ply] = (uint8_t)action;
        apply_legal(me, opp, action);
        player = -player;
        ++ply;
        over = game_over(me, opp, cells);
    }
    S.me[g] = me;
    S.opp[g] = opp;
    S.player[g] = (int8_t)player;
    S.ply[g] = ply;
    S.count_x[g] = 0;
    S.count_o[g] = 0;
    S.result[g] = BZ_MATCH_RUNNING;
    S.tree_of_game[g] = -1;
    if (over) match_finish(S, g, me, opp, player);
}

// a warp per game: the most visited root action of the game's tree, record, apply, terminal test, score
__global__ void __launch_bounds__(kThreads) match_advance_kernel(const bz_match_state S, const bz_tree_pools P, uint64_t cells) {
    const int g = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (g >= S.n_games) return;
    const int lane = threadIdx.x & 31;
    const int t = S.tree_of_game[g];
    if (t < 0) return;  // ended
    BZ_CHECK(t < P.n_trees && t < S.n_trees && S.game_of_tree[t] == g, 33);  // tree of the game
    const uint32_t rmeta = P.root_meta[t];
    const int n = (int)((rmeta >> BZ_META_N_SHIFT) & 63u);
    const uint32_t *blk = P.arena + (int64_t)t * P.arena_units * 8 + (int64_t)(rmeta >> BZ_META_OFF_SHIFT) * 8;
    int Ne = 0, N32 = 0;
    unsigned act = 127u, act32 = 127u;
    if (lane < n) {
        Ne = (int)blk[BZ_NODE_HEADER_WORDS + lane];
        act = blk[BZ_NODE_HEADER_WORDS + 3 * n + lane] & 127u;
    }
    if (n > 32) {
        N32 = (int)blk[BZ_NODE_HEADER_WORDS + 32];
        act32 = blk[BZ_NODE_HEADER_WORDS + 3 * n + 32] & 127u;
    }
    const int total = __reduce_add_sync(kFull, Ne) + N32;
    uint64_t me = S.me[g], opp = S.opp[g];
    const int player = S.player[g], ply = S.ply[g];
    unsigned action;
    if (n == 0 || total == 0) {  // a one-iteration search leaves no visits below the root: first legal move, or a pass
        const uint64_t m = legal_mask(me, opp, cells);
        action = m ? (unsigned)(__ffsll((long long)m) - 1) : 64u;
    } else {  // most visited, lowest action id on ties (selfplay_advance_kernel, best_action_kernel)
        unsigned key = (lane < n && Ne > 0) ? (((unsigned)Ne << 7) | (127u - act)) : 0u;
        if (n > 32 && N32 > 0) {
            const unsigned k32 = ((unsigned)N32 << 7) | (127u - act32);
            key = k32 > key ? k32 : key;
        }
        key = __reduce_max_sync(kFull, key);
        action = 127u - (key & 127u);
    }
    if (lane != 0) return;
    BZ_CHECK(ply >= 0 && ply < BZ_MATCH_MAX_PLIES && action <= 64u, 34);  // move row, action
    S.moves[(int64_t)g * BZ_MATCH_MAX_PLIES + ply] = (uint8_t)action;
    apply_legal(me, opp, action);  // the next mover's view
    S.me[g] = me;
    S.opp[g] = opp;
    S.player[g] = (int8_t)(-player);
    S.ply[g] = ply + 1;
    S.tree_of_game[g] = -1;  // the next layout assigns a tree again
    if (game_over(me, opp, cells) || ply + 1 >= BZ_MATCH_MAX_PLIES) match_finish(S, g, me, opp, -player);
}

// ---- tournaments ------------------------------------------------------------------------------------------------------
// Game pair i is pairing (first[i], second[i]): `first` is X in game 2i and O in game 2i+1.  The entrant to move in game g
// is its X-entrant when X is to move, the other one otherwise; -1 (BZ_CHECK) for an entrant id >= n_entrants.
__device__ __forceinline__ int tournament_entrant_to_move(const bz_tournament_state &S, int g) {
    const int i = g >> 1;
    const int a = S.first[i], b = S.second[i];
    const bool x_is_first = (g & 1) == 0, x_to_move = S.match.player[g] > 0;
    const int e = x_is_first == x_to_move ? a : b;
    BZ_CHECK(a < S.n_entrants && b < S.n_entrants, 35);  // entrant id
    return e < S.n_entrants ? e : -1;
}

// one CTA: stable partition of the live games by the entrant to move -- entrants in id order, games in game order inside
// an entrant, every non-empty range but the last padded with empty boards to the next multiple of 56 (a CTA pair of
// the one-launch search loads one entrant).  Ranks: __match_any_sync inside a warp, per-warp counts of each entrant in a
// 32 x E table scanned over the warps, a running base per entrant across the 1024-game chunks.
__global__ void __launch_bounds__(kLayoutThreads) tournament_layout_kernel(const bz_tournament_state S) {
    const bz_match_state &M = S.match;
    const int E = S.n_entrants;
    __shared__ unsigned cnt[BZ_MAX_ENTRANTS], start[BZ_MAX_ENTRANTS], pad_end[BZ_MAX_ENTRANTS];
    __shared__ unsigned wcnt[32][BZ_MAX_ENTRANTS];  // [warp][entrant]: movers, then the warp's first tree in the range
    __shared__ int n_search_s, last_s;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid < BZ_MAX_ENTRANTS) cnt[tid] = 0;
    __syncthreads();
    // pass 1: movers of each entrant
    for (int g = tid; g < M.n_games; g += kLayoutThreads) {
        if (M.result[g] != BZ_MATCH_RUNNING) continue;
        const int e = tournament_entrant_to_move(S, g);
        if (e >= 0) atomicAdd(&cnt[e], 1u);
    }
    __syncthreads();
    if (tid == 0) {
        int last = -1;
        for (int e = 0; e < E; ++e)
            if (cnt[e]) last = e;
        unsigned t = 0;
        for (int e = 0; e < E; ++e) {
            start[e] = t;
            t += cnt[e];
            if (cnt[e] && e != last) t = (t + kPairTrees - 1) / kPairTrees * kPairTrees;  // the next range: a pair boundary
            pad_end[e] = t;
        }
        n_search_s = (int)t;
        last_s = last;
    }
    __syncthreads();
    const int n_search = n_search_s, last = last_s;
    // pass 2: trees of the live games
    unsigned base_lo = 0, base_hi = 0;  // warp w: trees already given to entrants w and w + 32 by earlier chunks
    for (int g0 = 0; g0 < M.n_games; g0 += kLayoutThreads) {
        for (int k = tid; k < 32 * BZ_MAX_ENTRANTS; k += kLayoutThreads) (&wcnt[0][0])[k] = 0;
        __syncthreads();
        const int g = g0 + tid;
        const int e = g < M.n_games && M.result[g] == BZ_MATCH_RUNNING ? tournament_entrant_to_move(S, g) : -1;
        const unsigned same = __match_any_sync(kFull, e);
        const unsigned rank = __popc(same & ((1u << lane) - 1u));
        if (e >= 0 && rank == 0) wcnt[w][e] = __popc(same);
        __syncthreads();
        // warp w scans the column of entrants w and w + 32 over the 32 warps (lane = warp)
        for (int h = 0; h < 2; ++h) {
            const int ee = w + 32 * h;
            if (ee >= E) break;
            const unsigned v = wcnt[lane][ee];
            unsigned incl = v;
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned up = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += up;
            }
            unsigned &base = h ? base_hi : base_lo;
            wcnt[lane][ee] = start[ee] + base + incl - v;
            base += __shfl_sync(kFull, incl, 31);
        }
        __syncthreads();
        if (g < M.n_games) {
            int t = -1;
            if (e >= 0) {
                t = (int)(wcnt[w][e] + rank);
                BZ_CHECK(t >= 0 && t < n_search && n_search <= M.n_trees, 36);  // tree row
                M.game_of_tree[t] = g;
                M.root_me[t] = M.me[g];
                M.root_opp[t] = M.opp[g];
            }
            M.tree_of_game[g] = t;
        }
        __syncthreads();  // wcnt is cleared for the next chunk
    }
    // padding after each range but the last, and the rows past the searched prefix: empty boards (a finished game, no
    // move for either side: the search expands nothing there)
    for (int e = 0; e < E; ++e) {
        const int t = (int)(start[e] + cnt[e]) + tid;
        if (t < (int)pad_end[e]) {
            M.game_of_tree[t] = -1;
            M.root_me[t] = 0ull;
            M.root_opp[t] = 0ull;
        }
    }
    for (int t = n_search + tid; t < M.n_trees; t += kLayoutThreads) {
        M.game_of_tree[t] = -1;
        M.root_me[t] = 0ull;
        M.root_opp[t] = 0ull;
    }
    // the entrant of each CTA pair: the range that holds its first tree; pairs past the prefix: the last entrant
    const int n_pairs = (M.n_trees + kPairTrees - 1) / kPairTrees;
    for (int q = tid; q < n_pairs; q += kLayoutThreads) {
        int owner = last < 0 ? 0 : last;
        for (int e = 0; e < E; ++e)
            if (cnt[e] && (unsigned)(q * kPairTrees) >= start[e] && (unsigned)(q * kPairTrees) < pad_end[e]) owner = e;
        M.pair_net[q] = (uint8_t)owner;
    }
    if (tid == 0) {
        unsigned live = 0;
        for (int e = 0; e < E; ++e) live += cnt[e];
        M.counters[0] = live;
        M.counters[1] = n_search;
        M.counters[2] = n_search - (int)live;
    }
}

int check_match(const bz_match_state *s) {
    if (!s) return BZ_ERR_ARG;
    if (!(s->board_size == 4 || s->board_size == 6 || s->board_size == 8)) return BZ_ERR_ARG;
    if (s->n_games < 0 || (s->n_games & 1) || s->n_games >= (1 << 16) || s->opening_plies < 0 ||
        s->n_trees < s->n_games + kPairTrees - 1)
        return BZ_ERR_ARG;
    if (!s->me || !s->opp || !s->player || !s->ply || !s->result || !s->count_x || !s->count_o || !s->moves ||
        !s->tree_of_game || !s->game_of_tree || !s->root_me || !s->root_opp || !s->pair_net || !s->counters)
        return BZ_ERR_ARG;
    return BZ_OK;
}

int check_tournament(const bz_tournament_state *s) {
    if (!s) return BZ_ERR_ARG;
    const int rc = check_match(&s->match);
    if (rc != BZ_OK) return rc;
    if (s->n_entrants < 1 || s->n_entrants > BZ_MAX_ENTRANTS || !s->first || !s->second ||
        s->match.n_trees < s->match.n_games + (kPairTrees - 1) * (s->n_entrants - 1))
        return BZ_ERR_ARG;
    return BZ_OK;
}

int check_state(const bz_selfplay_state *s) {
    if (!s) return BZ_ERR_ARG;
    if (!(s->board_size == 4 || s->board_size == 6 || s->board_size == 8)) return BZ_ERR_ARG;
    if (s->n_games < 0 || s->max_plies < 2 || s->replay_cap < 0 || s->temp_plies < 0) return BZ_ERR_ARG;
    if (!s->me || !s->opp || !s->player || !s->ply || !s->game_id || !s->hist_me || !s->hist_opp || !s->hist_player ||
        !s->hist_action || !s->hist_pi || !s->rp_me || !s->rp_opp || !s->rp_pi || !s->rp_z || !s->rp_game ||
        !s->rp_ply || !s->counters)
        return BZ_ERR_ARG;
    return BZ_OK;
}

}  // namespace
}  // namespace bz

using namespace bz;

extern "C" {

int bz_selfplay_init(const bz_selfplay_state *st, int64_t first_game_id, bz_stream_t stream) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    const int n = st->n_games > 8 ? st->n_games : 8;
    selfplay_init_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(*st, first_game_id);
    return launch_rc();
}

int bz_selfplay_advance(const bz_selfplay_state *st, const bz_tree_pools *pools, uint8_t *action_out,
                        bz_stream_t stream) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    if (!pools || pools->game != BZ_GAME_REVERSI || pools->n_trees != st->n_games || pools->board_size != st->board_size ||
        !pools->root_meta || !pools->arena)
        return BZ_ERR_ARG;
    if (st->n_games == 0) return BZ_OK;
    selfplay_advance_kernel<<<(st->n_games + kWarpsPerCta - 1) / kWarpsPerCta, kThreads, 0, as_stream(stream)>>>(
        *st, *pools, action_out, cell_mask(st->board_size));
    return launch_rc();
}

int bz_match_init(const bz_match_state *st, bz_stream_t stream) {
    int rc = check_match(st);
    if (rc != BZ_OK) return rc;
    rc = cuda_rc(cudaMemsetAsync(st->counters, 0, 8 * sizeof(int64_t), as_stream(stream)));
    if (rc != BZ_OK || st->n_games == 0) return rc;
    match_init_kernel<<<(st->n_games + 255) / 256, 256, 0, as_stream(stream)>>>(*st, cell_mask(st->board_size));
    return launch_rc();
}

int bz_tournament_layout(const bz_tournament_state *st, bz_stream_t stream) {
    int rc = check_tournament(st);
    if (rc != BZ_OK) return rc;
    tournament_layout_kernel<<<1, kLayoutThreads, 0, as_stream(stream)>>>(*st);
    return launch_rc();
}

int bz_match_advance(const bz_match_state *st, const bz_tree_pools *pools, bz_stream_t stream) {
    int rc = check_match(st);
    if (rc != BZ_OK) return rc;
    if (!pools || pools->game != BZ_GAME_REVERSI || pools->n_trees != st->n_trees || pools->board_size != st->board_size ||
        !pools->root_meta || !pools->arena)
        return BZ_ERR_ARG;
    if (st->n_games == 0) return BZ_OK;
    match_advance_kernel<<<(st->n_games + kWarpsPerCta - 1) / kWarpsPerCta, kThreads, 0, as_stream(stream)>>>(
        *st, *pools, cell_mask(st->board_size));
    return launch_rc();
}

int bz_reversi_symmetry(const uint64_t *me, const uint64_t *opp, const float *pi, const uint8_t *sym,
                        uint64_t *me_out, uint64_t *opp_out, float *pi_out, int64_t n, int size,
                        bz_stream_t stream) {
    if (n < 0 || !(size == 4 || size == 6 || size == 8) ||
        (n && (!me || !opp || !pi || !sym || !me_out || !opp_out || !pi_out)))
        return BZ_ERR_ARG;
    if (me == me_out || opp == opp_out || pi == pi_out) return BZ_ERR_ARG;  // not an in-place transform
    if (n == 0) return BZ_OK;
    symmetry_kernel<<<persistent_grid(n * A, 256, 8), 256, 0, as_stream(stream)>>>(me, opp, pi, sym, me_out, opp_out,
                                                                                pi_out, n, size);
    return launch_rc();
}

int bz_record_hash(const uint64_t *me, const uint64_t *opp, const float *pi, uint64_t *hash_out, int64_t n, bz_stream_t stream) {
    if (n < 0 || (n && (!me || !opp || !pi || !hash_out))) return BZ_ERR_ARG;
    if (n == 0) return BZ_OK;
    record_hash_kernel<<<persistent_grid(n * 32, 256, 8), 256, 0, as_stream(stream)>>>(me, opp, pi, hash_out, n);
    return launch_rc();
}

int bz_philox_u32(uint64_t seed, const int64_t *game_id, const int32_t *ply, uint32_t *out, int64_t n,
                  bz_stream_t stream) {
    if (n < 0 || (n && (!game_id || !ply || !out))) return BZ_ERR_ARG;
    if (n == 0) return BZ_OK;
    philox_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(seed, game_id, ply, out, n);
    return launch_rc();
}

}  // extern "C"

#ifdef BZ_BOUNDS_CHECK
// debug builds: [code of the first failed check, block, thread, violations] of the self-play kernels; clears the record
extern "C" int bz_debug_checks_selfplay(int *host_out) {
    int rc = bz::cuda_rc(cudaMemcpyFromSymbol(host_out, bz::g_bz_check, sizeof(int) * 4));
    if (rc) return rc;
    const int zero[4] = {0, 0, 0, 0};
    return bz::cuda_rc(cudaMemcpyToSymbol(bz::g_bz_check, zero, sizeof(zero)));
}
#endif
