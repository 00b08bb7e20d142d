// Lockstep self-play driver kernels for sm_100a: the batched form of the reference episode loop
// (src/reversi/game_logic/reversi_terminal.py:16-38): after a search, every game slot picks its
// move from the root visit counts, records (board, pi), applies the move (or pass), tests for the
// end of the game (reversi_board.py:61-65), scores finished games (get_score, :67-76), flushes
// them to the replay buffer and restarts the slot.  One warp per game slot == per tree.
#include "bitboard.cuh"
#include "common.cuh"
#include "minimax.cuh"

namespace bz {
namespace {

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kWarpsPerCta = 4;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int A = BZ_REVERSI_ACTIONS;

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

// the game of slot s has left it (finished, or handed over to the endgame queue): the start position, the next game id
__device__ __forceinline__ void restart_slot(const bz_selfplay_state &S, int s, int64_t gid) {
    S.me[s] = start_me(S.board_size);
    S.opp[s] = start_opp(S.board_size);
    S.player[s] = 1;
    S.ply[s] = 0;
    S.game_id[s] = gid + S.id_stride;
}

// the result of a game that has ended at (me, opp), seen by the side to move after `player`'s last move (get_score: more
// discs wins); absolute: +1 X, -1 O, 0 draw
__device__ __forceinline__ int disc_winner(uint64_t me, uint64_t opp, int player) {
    const int cm = __popcll(me), co = __popcll(opp);
    return ((cm > co) - (cm < co)) * (-player);
}

// game g is audited (never resigns) iff philox_u32(seed, g, 0xFFFFFFFF) < audit_below: the counter is never a ply
__device__ __forceinline__ bool resign_audited(uint64_t seed, int64_t gid, uint64_t audit_below) {
    return (uint64_t)philox_u32(seed, (uint64_t)gid, 0xFFFFFFFFu) < audit_below;
}

// the ply `ply` of game `gid` is searched with the full budget iff philox_u32(seed, gid, 0x80000000 | ply) < full_below:
// the counter is never a ply (< 128) and never the audit draw's 0xFFFFFFFF
__device__ __forceinline__ bool cap_full(uint64_t seed, int64_t gid, int ply, uint64_t full_below) {
    return (uint64_t)philox_u32(seed, (uint64_t)gid, 0x80000000u | (uint32_t)ply) < full_below;
}

// a warp: the game `gid` has ended with `winner` (absolute: +1 X, -1 O, 0 draw); copy its nrec history rows, block `block`
// of max_plies rows in hist_*, to the replay buffer (whole or not at all); lane 0 counts.  kResign: the q rows (hist_q)
// go to R->rp_q as well, and an audited game is counted in R->counters[1].  kCap: the flag rows (hist_full) go to
// Cs->rp_full.
template <bool kResign = false, bool kCap = false>
__device__ __forceinline__ void flush_game(const bz_selfplay_state &S, const uint64_t *hist_me, const uint64_t *hist_opp,
                                           const int8_t *hist_player, const float *hist_pi, int block, int max_plies,
                                           int nrec, int64_t gid, int winner, int lane,
                                           const bz_selfplay_resign_state *R = nullptr, const float *hist_q = nullptr,
                                           const bz_selfplay_cap_state *Cs = nullptr, const uint8_t *hist_full = nullptr) {
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
        if constexpr (kResign) {
            if (resign_audited(S.seed, gid, R->audit_below)) atomicAdd(&R->counters[1], 1ull);
        }
    }
    rb = __shfl_sync(kFull, rb, 0);
    __syncwarp();  // the record written above is visible to the copying lanes
    const int64_t h0 = (int64_t)block * max_plies;
    if (rb != ~0ull) {
        BZ_CHECK(rb + (unsigned long long)nrec <= (unsigned long long)S.replay_cap && nrec <= S.max_plies, 22);  // replay rows
        for (int r = lane; r < nrec; r += 32) {
            S.rp_me[rb + r] = hist_me[h0 + r];
            S.rp_opp[rb + r] = hist_opp[h0 + r];
            S.rp_z[rb + r] = (int8_t)(winner * hist_player[h0 + r]);
            S.rp_game[rb + r] = gid;
            S.rp_ply[rb + r] = (int16_t)r;
            if constexpr (kResign) R->rp_q[rb + r] = hist_q[h0 + r];
            if constexpr (kCap) Cs->rp_full[rb + r] = hist_full[h0 + r];
        }
        const int64_t nf = (int64_t)nrec * A;  // pi rows are contiguous in both buffers
        const float *src = hist_pi + h0 * A;
        float *dst = S.rp_pi + (int64_t)rb * A;
        for (int64_t i = lane; i < nf; i += 32) dst[i] = src[i];
    } else if (lane == 0) {
        atomicAdd(&S.counters[5], (unsigned long long)nrec);
    }
}

// a warp: move the game of slot s -- (me, opp) with `player` to move, nrec history rows -- to the next free entry of the
// endgame queue, its rows to the entry's history block (row == entry: the queue fills from an empty state between solver
// phases); false, and counted, when the queue is full.  kResign: the q rows go to R->eg_hist_q as well.  kCap: the flag
// rows go to Cs->eg_hist_full.
template <bool kResign, bool kCap = false>
__device__ __forceinline__ bool handover(const bz_selfplay_state &S, const bz_selfplay_endgame_state &EG, int s, int lane,
                                         uint64_t me, uint64_t opp, int player, int nrec, int64_t gid,
                                         const bz_selfplay_resign_state *R, const bz_selfplay_cap_state *Cs = nullptr) {
    int q = -1;
    if (lane == 0) {
        int cur = *EG.count;
        while (cur < EG.cap) {
            const int seen = atomicCAS(EG.count, cur, cur + 1);
            if (seen == cur) {
                q = cur;
                break;
            }
            cur = seen;
        }
        if (q < 0) atomicAdd(&EG.counters[2], 1ull);
    }
    q = __shfl_sync(kFull, q, 0);
    if (q < 0) return false;
    BZ_CHECK(q < EG.cap && nrec <= EG.max_plies && nrec <= S.max_plies, 23);  // queue entry, history rows
    __syncwarp();  // the record written above is visible to the copying lanes
    const int64_t src = (int64_t)s * S.max_plies, dst = (int64_t)q * EG.max_plies;
    for (int r = lane; r < nrec; r += 32) {
        EG.hist_me[dst + r] = S.hist_me[src + r];
        EG.hist_opp[dst + r] = S.hist_opp[src + r];
        EG.hist_player[dst + r] = S.hist_player[src + r];
        EG.hist_action[dst + r] = S.hist_action[src + r];
        if constexpr (kResign) R->eg_hist_q[dst + r] = R->hist_q[src + r];
        if constexpr (kCap) Cs->eg_hist_full[dst + r] = Cs->hist_full[src + r];
    }
    const int64_t nf = (int64_t)nrec * A;
    for (int64_t i = lane; i < nf; i += 32) EG.hist_pi[dst * A + i] = S.hist_pi[src * A + i];
    if (lane == 0) {
        EG.me[q] = me;
        EG.opp[q] = opp;
        EG.player[q] = (int8_t)player;
        EG.ply[q] = nrec;
        EG.game_id[q] = gid;
        EG.row[q] = q;
        atomicAdd(&S.counters[1], 1ull);
        atomicAdd(&EG.counters[0], 1ull);
    }
    return true;
}

// a warp: the most visited root action, lowest action id on ties (players.py:92-98 applied to visit counts); lane i holds
// edge i (Ne, act), edge 32 is held uniformly (N32, act32)
__device__ __forceinline__ unsigned greedy_action(int Ne, unsigned act, int N32, unsigned act32, int n, int lane) {
    unsigned key = (lane < n && Ne > 0) ? (((unsigned)Ne << 7) | (127u - act)) : 0u;
    if (n > 32 && N32 > 0) {
        const unsigned k32 = ((unsigned)N32 << 7) | (127u - act32);
        key = k32 > key ? k32 : key;
    }
    key = __reduce_max_sync(kFull, key);
    return 127u - (key & 127u);
}

// a warp per game slot: the move from the root visit counts, the record, the move applied, the terminal test; a finished
// game is flushed and its slot restarts.  kEndgame: a game whose move leaves EG->empties empties or fewer for the first
// time goes to the endgame queue instead (and its slot restarts) when the queue has room.  kResign: the ply's q (W / N of
// the most visited root edge, the mover's view) is recorded, and a game that is not audited resigns when q < threshold:
// the record is kept, the mover loses, the game is flushed and the slot restarts before the move is applied.  kCap: the
// search of slot s is tree Cs->tree_of_slot[s] of the pools, and the ply's flag (full or fast) goes to Cs->hist_full.
template <bool kEndgame, bool kResign = false, bool kCap = false>
__device__ __forceinline__ void advance_slot(const bz_selfplay_state &S, const bz_tree_pools &P, uint8_t *action_out,
                                             uint64_t cells, const bz_selfplay_endgame_state *EG, int s, int lane,
                                             const bz_selfplay_resign_state *R = nullptr,
                                             const bz_selfplay_cap_state *Cs = nullptr) {

    // root statistics: lane i holds edge i (ascending action id); a 33rd edge is read uniformly
    int tree = s;
    if constexpr (kCap) {
        tree = Cs->tree_of_slot[s];
        BZ_CHECK(tree >= 0 && tree < P.n_trees, 26);  // tree of the slot
    }
    const uint32_t rmeta = P.root_meta[tree];
    const int n = (int)((rmeta >> BZ_META_N_SHIFT) & 63u);
    const uint32_t *blk = P.arena + (int64_t)tree * P.arena_units * 8 + (int64_t)(rmeta >> BZ_META_OFF_SHIFT) * 8;
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

    // --- q of the ply (kResign): W / N of the greedy pick a*, whether or not the move is sampled; NaN without visits ----
    [[maybe_unused]] unsigned best = 0u;
    [[maybe_unused]] float q = __int_as_float(0x7FC00000);
    if constexpr (kResign) {
        if (n > 0 && total > 0) {
            best = greedy_action(Ne, act, N32, act32, n, lane);
            const unsigned hit = __ballot_sync(kFull, lane < n && act == best);
            const int src = hit ? __ffs(hit) - 1 : 0;
            float w = 0.f;
            if (hit && lane == src) w = __uint_as_float(blk[BZ_NODE_HEADER_WORDS + n + lane]);
            w = __shfl_sync(kFull, w, src);
            int nb = __shfl_sync(kFull, Ne, src);
            if (!hit) {  // a* is edge 32
                w = __uint_as_float(blk[BZ_NODE_HEADER_WORDS + n + 32]);
                nb = N32;
            }
            q = __fdiv_rn(w, (float)nb);
        }
    }

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
    } else if constexpr (kResign) {
        action = best;
    } else {
        action = greedy_action(Ne, act, N32, act32, n, lane);
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
        if constexpr (kResign) R->hist_q[h] = q;
        if constexpr (kCap) Cs->hist_full[h] = (uint8_t)cap_full(S.seed, gid, ply, Cs->full_below);
    }

    // --- resignation (kResign): before the move is applied, so before the handover test; NaN never compares below -----
    if constexpr (kResign) {
        if (q < R->threshold && !resign_audited(S.seed, gid, R->audit_below)) {
            flush_game<true, kCap>(S, S.hist_me, S.hist_opp, S.hist_player, S.hist_pi, s, S.max_plies, ply + 1, gid,
                                   -player, lane, R, R->hist_q, Cs, kCap ? Cs->hist_full : nullptr);
            if (lane == 0) {
                atomicAdd(&R->counters[0], 1ull);
                restart_slot(S, s, gid);
            }
            return;
        }
    }

    // --- apply, terminal test -----------------------------------------------------------------
    [[maybe_unused]] const uint64_t occupied = me | opp;
    apply_legal(me, opp, action);  // now the NEXT mover's view; next player = -player
    const bool over = (legal_mask(me, opp, cells) | legal_mask(opp, me, cells)) == 0;
    const int nrec = ply + 1;
    if (!over && nrec < S.max_plies) {
        if constexpr (kEndgame) {
            // the first position at E empties or fewer (the move placed a disc): a game the full queue refuses is not
            // offered again and is searched to its end
            if (__popcll(cells) - __popcll(me | opp) <= EG->empties && EG->empties < __popcll(cells) - __popcll(occupied) &&
                handover<kResign, kCap>(S, *EG, s, lane, me, opp, -player, nrec, gid, R, Cs)) {
                if (lane == 0) restart_slot(S, s, gid);
                return;
            }
        }
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
    flush_game<kResign, kCap>(S, S.hist_me, S.hist_opp, S.hist_player, S.hist_pi, s, S.max_plies, nrec, gid,
                              disc_winner(me, opp, player), lane, R, kResign ? R->hist_q : nullptr, Cs,
                              kCap ? Cs->hist_full : nullptr);
    if (lane == 0) restart_slot(S, s, gid);
}

__global__ void __launch_bounds__(kThreads)
    selfplay_advance_kernel(const bz_selfplay_state S, const bz_tree_pools P, uint8_t *action_out, uint64_t cells) {
    const int s = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (s >= S.n_games) return;
    advance_slot<false>(S, P, action_out, cells, nullptr, s, threadIdx.x & 31);
}

__global__ void __launch_bounds__(kThreads)
    selfplay_advance_endgame_kernel(const bz_selfplay_state S, const bz_tree_pools P, uint8_t *action_out, uint64_t cells,
                                    const __grid_constant__ bz_selfplay_endgame_state EG) {
    const int s = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (s >= S.n_games) return;
    advance_slot<true>(S, P, action_out, cells, &EG, s, threadIdx.x & 31);
}

// kEndgame = false: EG is not read
template <bool kEndgame>
__global__ void __launch_bounds__(kThreads)
    selfplay_advance_resign_kernel(const bz_selfplay_state S, const bz_tree_pools P, uint8_t *action_out, uint64_t cells,
                                   const __grid_constant__ bz_selfplay_endgame_state EG,
                                   const __grid_constant__ bz_selfplay_resign_state R) {
    const int s = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (s >= S.n_games) return;
    advance_slot<kEndgame, true>(S, P, action_out, cells, &EG, s, threadIdx.x & 31, &R);
}

// kEndgame = false: EG is not read; kResign = false: R is not read
template <bool kEndgame, bool kResign>
__global__ void __launch_bounds__(kThreads)
    selfplay_advance_cap_kernel(const bz_selfplay_state S, const bz_tree_pools P, uint8_t *action_out, uint64_t cells,
                                const __grid_constant__ bz_selfplay_endgame_state EG,
                                const __grid_constant__ bz_selfplay_resign_state R,
                                const __grid_constant__ bz_selfplay_cap_state Cs) {
    const int s = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (s >= S.n_games) return;
    advance_slot<kEndgame, kResign, true>(S, P, action_out, cells, &EG, s, threadIdx.x & 31, &R, &Cs);
}

// ---- the endgame queue: one solver ply of every pending game -----------------------------------------------------------
// a warp per entry i < count: record the position with pi = 1/k on each of the k moves whose value is the root value
// (a forced pass: one-hot on 64), play the solver's first best move, flush a finished game (ply = -1 marks the entry).
// kResign: the record's q is NaN, and the flush carries the q rows (R->eg_hist_q) to the replay buffer.  kCap: the
// record's flag is 1 (an exact label), and the flush carries the flag rows (Cs->eg_hist_full).
template <bool kResign, bool kCap>
__device__ __forceinline__ void endgame_ply(const bz_selfplay_state &S, const bz_selfplay_endgame_state &EG, int i,
                                            int lane, const uint8_t *solve_action, const int8_t *solve_value,
                                            const int8_t *move_value, uint64_t cells, const bz_selfplay_resign_state *R,
                                            const bz_selfplay_cap_state *Cs) {
    const int ply = EG.ply[i], player = EG.player[i], b = EG.row[i];
    const int64_t gid = EG.game_id[i];
    uint64_t me = EG.me[i], opp = EG.opp[i];
    const unsigned action = solve_action[i];
    const int v = solve_value[i];
    const int8_t *mv = move_value + (int64_t)i * A;
    const bool o0 = mv[lane] == v, o1 = mv[lane + 32] == v, o64 = mv[64] == v;  // illegal actions hold -128 < any value
    const int k = __popc(__ballot_sync(kFull, o0)) + __popc(__ballot_sync(kFull, o1)) + (o64 ? 1 : 0);
    const int64_t h = (int64_t)b * EG.max_plies + ply;
    BZ_CHECK(i < EG.cap && b >= 0 && b < EG.cap && ply >= 0 && ply < EG.max_plies && action <= 64u && k >= 1, 24);
    const float p = __fdiv_rn(1.0f, (float)(k > 0 ? k : 1));
    float *pi = EG.hist_pi + h * A;
    pi[lane] = o0 ? p : 0.f;
    pi[lane + 32] = o1 ? p : 0.f;
    if (lane == 0) {
        pi[64] = o64 ? p : 0.f;
        EG.hist_me[h] = me;
        EG.hist_opp[h] = opp;
        EG.hist_player[h] = (int8_t)player;
        EG.hist_action[h] = (uint8_t)action;
        if constexpr (kResign) R->eg_hist_q[h] = __int_as_float(0x7FC00000);
        if constexpr (kCap) Cs->eg_hist_full[h] = 1;
        atomicAdd(&EG.counters[1], 1ull);
    }
    apply_legal(me, opp, action);  // the next mover's view
    const bool over = (legal_mask(me, opp, cells) | legal_mask(opp, me, cells)) == 0;
    const int nrec = ply + 1;
    if (!over && nrec < EG.max_plies) {
        if (lane == 0) {
            EG.me[i] = me;
            EG.opp[i] = opp;
            EG.player[i] = (int8_t)(-player);
            EG.ply[i] = nrec;
            atomicAdd(&S.counters[1], 1ull);
        }
        return;
    }
    flush_game<kResign, kCap>(S, EG.hist_me, EG.hist_opp, EG.hist_player, EG.hist_pi, b, EG.max_plies, nrec, gid,
                              disc_winner(me, opp, player), lane, R, R->eg_hist_q, Cs, kCap ? Cs->eg_hist_full : nullptr);
    if (lane == 0) {
        EG.ply[i] = -1;
        atomicAdd(&EG.counters[3], 1ull);
    }
}

template <bool kResign>
__global__ void __launch_bounds__(kThreads)
    endgame_ply_kernel(const bz_selfplay_state S, const __grid_constant__ bz_selfplay_endgame_state EG,
                       const uint8_t *solve_action, const int8_t *solve_value, const int8_t *move_value, uint64_t cells,
                       const __grid_constant__ bz_selfplay_resign_state R) {
    const int i = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (i >= *EG.count) return;
    endgame_ply<kResign, false>(S, EG, i, threadIdx.x & 31, solve_action, solve_value, move_value, cells, &R, nullptr);
}

// kResign = false: R is not read
template <bool kResign>
__global__ void __launch_bounds__(kThreads)
    endgame_ply_cap_kernel(const bz_selfplay_state S, const __grid_constant__ bz_selfplay_endgame_state EG,
                           const uint8_t *solve_action, const int8_t *solve_value, const int8_t *move_value,
                           uint64_t cells, const __grid_constant__ bz_selfplay_resign_state R,
                           const __grid_constant__ bz_selfplay_cap_state Cs) {
    const int i = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (i >= *EG.count) return;
    endgame_ply<kResign, true>(S, EG, i, threadIdx.x & 31, solve_action, solve_value, move_value, cells, &R, &Cs);
}

// one CTA: the live entries (ply >= 0) of [0, count) to the front, in order; count = their number.  In place: a chunk's
// entries are read before any of them is written, and every entry moves down, never into a later chunk.
__global__ void __launch_bounds__(1024) endgame_compact_kernel(const __grid_constant__ bz_selfplay_endgame_state EG) {
    __shared__ int warp_base[32];
    __shared__ int chunk_live;
    const int n = *EG.count;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    int carry = 0;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + tid;
        const bool live = i < n && EG.ply[i] >= 0;
        uint64_t me = 0, opp = 0;
        int64_t gid = 0;
        int ply = 0, row = 0, player = 0;
        if (live) {
            me = EG.me[i];
            opp = EG.opp[i];
            gid = EG.game_id[i];
            ply = EG.ply[i];
            row = EG.row[i];
            player = EG.player[i];
        }
        const unsigned bal = __ballot_sync(kFull, live);
        if (lane == 0) warp_base[w] = __popc(bal);
        __syncthreads();
        if (w == 0) {
            const int c = warp_base[lane];
            int incl = c;
            for (int d = 1; d < 32; d <<= 1) {
                const int up = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += up;
            }
            warp_base[lane] = incl - c;
            if (lane == 31) chunk_live = incl;
        }
        __syncthreads();
        if (live) {
            const int d = carry + warp_base[w] + __popc(bal & ((1u << lane) - 1u));
            BZ_CHECK(d <= i && d < EG.cap, 25);  // entries move down
            EG.me[d] = me;
            EG.opp[d] = opp;
            EG.game_id[d] = gid;
            EG.ply[d] = ply;
            EG.row[d] = row;
            EG.player[d] = (int8_t)player;
        }
        carry += chunk_live;
        __syncthreads();
    }
    __syncthreads();  // every thread has read count
    if (tid == 0) *EG.count = carry;
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
        if (m) action = pick_move(m, philox_u32(S.seed, pair_id, (uint32_t)ply));
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
// Tournaments with minimax entrants: the game of a tree whose CTA pair's entrant is in `minimax_entrants` (a bit per
// entrant) plays minimax_action[t] instead.
__global__ void __launch_bounds__(kThreads) match_advance_kernel(const bz_match_state S, const bz_tree_pools P, uint64_t cells,
                                                                 uint64_t minimax_entrants, const uint8_t *minimax_action) {
    const int g = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (g >= S.n_games) return;
    const int lane = threadIdx.x & 31;
    const int t = S.tree_of_game[g];
    if (t < 0) return;  // ended
    BZ_CHECK(t < S.n_trees && S.game_of_tree[t] == g, 33);  // tree of the game
    uint64_t me = S.me[g], opp = S.opp[g];
    const int player = S.player[g], ply = S.ply[g];
    unsigned action;
    if (minimax_entrants && ((minimax_entrants >> (S.pair_net[t / kPairTrees] & 63)) & 1)) {
        action = minimax_action[t];
        BZ_CHECK(action <= 64u, 37);  // a minimax move of a live game
    } else {  // a net entrant: the most visited root action
        BZ_CHECK(t < P.n_trees, 33);  // tree of the game
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

// ---- self-play with randomized search budgets ----------------------------------------------------------------------------
// one CTA: a two-key stable partition of the slots -- full slots (cap_full) to trees [0, n_full) in slot order, fast slots
// to [fast0, fast0 + n_fast) in slot order, fast0 = n_full rounded up to a CTA pair (56 trees); empty boards (a finished
// game: the search expands nothing there) on the padding [n_full, fast0) and after the fast range.  Ranks: ballots inside
// a warp, the per-warp counts scanned by warp 0, a running base per key across the 512-slot chunks.  512 threads: the
// Philox draw and the two running bases fit in registers without a spill.
constexpr int kCapLayoutThreads = 512, kCapLayoutWarps = kCapLayoutThreads / 32;
__global__ void __launch_bounds__(kCapLayoutThreads)
    selfplay_cap_layout_kernel(const bz_selfplay_state S, const __grid_constant__ bz_selfplay_cap_state Cs) {
    __shared__ unsigned wfull[kCapLayoutWarps], wfast[kCapLayoutWarps];  // [warp]: slots of the chunk, then the warp's first rank
    __shared__ unsigned sum_full, sum_fast;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    // pass 1: full slots
    unsigned mine = 0;
    for (int s = tid; s < S.n_games; s += kCapLayoutThreads)
        mine += cap_full(S.seed, S.game_id[s], S.ply[s], Cs.full_below);
    mine = __reduce_add_sync(kFull, mine);
    if (lane == 0) wfull[w] = mine;
    __syncthreads();
    if (w == 0) {
        const unsigned v = __reduce_add_sync(kFull, lane < kCapLayoutWarps ? wfull[lane] : 0u);
        if (lane == 0) sum_full = v;
    }
    __syncthreads();
    const int n_full = (int)sum_full, n_fast = S.n_games - n_full;
    const int fast0 = (n_full + kPairTrees - 1) / kPairTrees * kPairTrees;
    // pass 2: trees of the slots
    int base_full = 0, base_fast = fast0;
    for (int s0 = 0; s0 < S.n_games; s0 += kCapLayoutThreads) {
        const int s = s0 + tid;
        const bool live = s < S.n_games;
        const bool full = live && cap_full(S.seed, S.game_id[s], S.ply[s], Cs.full_below);
        const unsigned bf = __ballot_sync(kFull, full), bs = __ballot_sync(kFull, live && !full);
        __syncthreads();  // the previous chunk's ranks have been read
        if (lane == 0) {
            wfull[w] = __popc(bf);
            wfast[w] = __popc(bs);
        }
        __syncthreads();
        if (w == 0) {
            const unsigned vf = lane < kCapLayoutWarps ? wfull[lane] : 0u, vs = lane < kCapLayoutWarps ? wfast[lane] : 0u;
            unsigned inf = vf, ins = vs;
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned uf = __shfl_up_sync(kFull, inf, d), us = __shfl_up_sync(kFull, ins, d);
                if (lane >= d) {
                    inf += uf;
                    ins += us;
                }
            }
            if (lane < kCapLayoutWarps) {
                wfull[lane] = inf - vf;
                wfast[lane] = ins - vs;
            }
            if (lane == 31) {
                sum_full = inf;
                sum_fast = ins;
            }
        }
        __syncthreads();
        if (live) {
            const unsigned below = (1u << lane) - 1u;
            const int t = full ? base_full + (int)(wfull[w] + __popc(bf & below))
                               : base_fast + (int)(wfast[w] + __popc(bs & below));
            BZ_CHECK(t >= 0 && t < Cs.n_trees && (full ? t < n_full : t >= fast0 && t < fast0 + n_fast), 27);  // tree row
            Cs.tree_of_slot[s] = t;
            Cs.root_me[t] = S.me[s];
            Cs.root_opp[t] = S.opp[s];
        }
        base_full += (int)sum_full;
        base_fast += (int)sum_fast;
    }
    for (int t = n_full + tid; t < fast0; t += kCapLayoutThreads) {
        Cs.root_me[t] = 0ull;
        Cs.root_opp[t] = 0ull;
    }
    for (int t = fast0 + n_fast + tid; t < Cs.n_trees; t += kCapLayoutThreads) {
        Cs.root_me[t] = 0ull;
        Cs.root_opp[t] = 0ull;
    }
    const int n_pairs = (Cs.n_trees + kPairTrees - 1) / kPairTrees;
    for (int q = tid; q < n_pairs; q += kCapLayoutThreads) Cs.pair_entrant[q] = q * kPairTrees < fast0 ? 0 : 1;
    if (tid == 0) {
        Cs.counters[0] += (unsigned long long)n_full;
        Cs.counters[1] += (unsigned long long)n_fast;
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

int check_endgame(const bz_selfplay_state *s, const bz_selfplay_endgame_state *e) {
    if (!e) return BZ_ERR_ARG;
    const int cells = s->board_size * s->board_size;
    if (e->empties < 1 || e->empties > BZ_SOLVE_MAX_EMPTIES || e->empties > cells - 5) return BZ_ERR_ARG;
    if (e->cap < 1 || e->cap > (1 << 22) || e->max_plies != s->max_plies) return BZ_ERR_ARG;
    if (!e->me || !e->opp || !e->player || !e->ply || !e->game_id || !e->row || !e->hist_me || !e->hist_opp ||
        !e->hist_player || !e->hist_action || !e->hist_pi || !e->count || !e->counters)
        return BZ_ERR_ARG;
    return BZ_OK;
}

int check_resign(const bz_selfplay_endgame_state *e, const bz_selfplay_resign_state *r) {
    if (!r) return BZ_ERR_ARG;
    if (!(r->threshold >= -1.0f && r->threshold <= 1.0f)) return BZ_ERR_ARG;  // NaN fails both
    if (r->audit_below > (1ull << 32)) return BZ_ERR_ARG;
    if (!r->hist_q || !r->rp_q || !r->counters || (e && !r->eg_hist_q)) return BZ_ERR_ARG;
    return BZ_OK;
}

int check_cap(const bz_selfplay_state *s, const bz_selfplay_endgame_state *e, const bz_selfplay_cap_state *c) {
    if (!c) return BZ_ERR_ARG;
    if (c->full_below > (1ull << 32)) return BZ_ERR_ARG;
    if (c->n_trees < s->n_games + kPairTrees - 1) return BZ_ERR_ARG;
    if (!c->tree_of_slot || !c->root_me || !c->root_opp || !c->pair_entrant || !c->hist_full || !c->rp_full ||
        !c->counters || (e && !c->eg_hist_full))
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

int bz_selfplay_advance_endgame(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg,
                                const bz_tree_pools *pools, uint8_t *action_out, bz_stream_t stream) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    rc = check_endgame(st, eg);
    if (rc != BZ_OK) return rc;
    if (!pools || pools->game != BZ_GAME_REVERSI || pools->n_trees != st->n_games || pools->board_size != st->board_size ||
        !pools->root_meta || !pools->arena)
        return BZ_ERR_ARG;
    if (st->n_games == 0) return BZ_OK;
    selfplay_advance_endgame_kernel<<<(st->n_games + kWarpsPerCta - 1) / kWarpsPerCta, kThreads, 0, as_stream(stream)>>>(
        *st, *pools, action_out, cell_mask(st->board_size), *eg);
    return launch_rc();
}

int bz_selfplay_advance_resign(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg,
                               const bz_selfplay_resign_state *rs, const bz_tree_pools *pools, uint8_t *action_out,
                               bz_stream_t stream) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    if (eg && (rc = check_endgame(st, eg)) != BZ_OK) return rc;
    rc = check_resign(eg, rs);
    if (rc != BZ_OK) return rc;
    if (!pools || pools->game != BZ_GAME_REVERSI || pools->n_trees != st->n_games || pools->board_size != st->board_size ||
        !pools->root_meta || !pools->arena)
        return BZ_ERR_ARG;
    if (st->n_games == 0) return BZ_OK;
    const unsigned grid = (st->n_games + kWarpsPerCta - 1) / kWarpsPerCta;
    const uint64_t cells = cell_mask(st->board_size);
    if (eg) {
        selfplay_advance_resign_kernel<true><<<grid, kThreads, 0, as_stream(stream)>>>(*st, *pools, action_out, cells, *eg,
                                                                                      *rs);
    } else {
        const bz_selfplay_endgame_state none = {};
        selfplay_advance_resign_kernel<false><<<grid, kThreads, 0, as_stream(stream)>>>(*st, *pools, action_out, cells, none,
                                                                                       *rs);
    }
    return launch_rc();
}

// the solve's workspace, then its action [cap], value [cap] and move values [cap, 65], each 16-byte aligned
static int64_t endgame_play_align16(int64_t b) { return (b + 15) & ~(int64_t)15; }

int64_t bz_selfplay_endgame_workspace_bytes(int64_t cap) {
    if (cap < 1) return 0;
    return endgame_play_align16(endgame_workspace_bytes(cap)) + 2 * endgame_play_align16(cap) +
           endgame_play_align16(cap * A);
}

// rs: NULL without resignation; cs: NULL without randomized budgets
static int endgame_play(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg,
                        const bz_selfplay_resign_state *rs, void *workspace, bool wld, bz_stream_t stream,
                        const bz_selfplay_cap_state *cs = nullptr) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    rc = check_endgame(st, eg);
    if (rc != BZ_OK) return rc;
    if (rs && (rc = check_resign(eg, rs)) != BZ_OK) return rc;
    if (cs && (rc = check_cap(st, eg, cs)) != BZ_OK) return rc;
    if (!workspace) return BZ_ERR_ARG;
    if (!aligned16(workspace)) return BZ_ERR_UNALIGNED;
    const int64_t cap = eg->cap;
    char *p = static_cast<char *>(workspace) + endgame_play_align16(endgame_workspace_bytes(cap));
    uint8_t *action = reinterpret_cast<uint8_t *>(p);
    int8_t *value = reinterpret_cast<int8_t *>(p + endgame_play_align16(cap));
    int8_t *move_value = value + endgame_play_align16(cap);
    const cudaStream_t s = as_stream(stream);
    const uint64_t cells = cell_mask(st->board_size);
    for (int k = 0; k < 2 * eg->empties; ++k) {
        rc = endgame_launch_live(eg->me, eg->opp, cap, eg->count, st->board_size, workspace, action, value, move_value, wld,
                                 s);
        if (rc != BZ_OK) return rc;
        const unsigned grid = (unsigned)((cap + kWarpsPerCta - 1) / kWarpsPerCta);
        if (cs) {
            const bz_selfplay_resign_state none = {};
            if (rs) {
                endgame_ply_cap_kernel<true><<<grid, kThreads, 0, s>>>(*st, *eg, action, value, move_value, cells, *rs, *cs);
            } else {
                endgame_ply_cap_kernel<false><<<grid, kThreads, 0, s>>>(*st, *eg, action, value, move_value, cells, none,
                                                                       *cs);
            }
        } else if (rs) {
            endgame_ply_kernel<true><<<grid, kThreads, 0, s>>>(*st, *eg, action, value, move_value, cells, *rs);
        } else {
            const bz_selfplay_resign_state none = {};
            endgame_ply_kernel<false><<<grid, kThreads, 0, s>>>(*st, *eg, action, value, move_value, cells, none);
        }
        endgame_compact_kernel<<<1, 1024, 0, s>>>(*eg);
        rc = launch_rc();
        if (rc != BZ_OK) return rc;
    }
    return BZ_OK;
}

int bz_selfplay_endgame_play(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg, void *workspace,
                             bz_stream_t stream) {
    return endgame_play(st, eg, nullptr, workspace, false, stream);
}

int bz_selfplay_endgame_play_wld(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg, void *workspace,
                                 bz_stream_t stream) {
    return endgame_play(st, eg, nullptr, workspace, true, stream);
}

int bz_selfplay_endgame_play_resign(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg,
                                    const bz_selfplay_resign_state *rs, void *workspace, int wld, bz_stream_t stream) {
    if (!rs) return BZ_ERR_ARG;
    return endgame_play(st, eg, rs, workspace, wld != 0, stream);
}

int bz_selfplay_endgame_play_cap(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg,
                                 const bz_selfplay_resign_state *rs, const bz_selfplay_cap_state *cs, void *workspace,
                                 int wld, bz_stream_t stream) {
    if (!cs) return BZ_ERR_ARG;
    return endgame_play(st, eg, rs, workspace, wld != 0, stream, cs);
}

int bz_selfplay_cap_layout(const bz_selfplay_state *st, const bz_selfplay_cap_state *cs, bz_stream_t stream) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    rc = check_cap(st, nullptr, cs);
    if (rc != BZ_OK) return rc;
    selfplay_cap_layout_kernel<<<1, kCapLayoutThreads, 0, as_stream(stream)>>>(*st, *cs);
    return launch_rc();
}

int bz_selfplay_advance_cap(const bz_selfplay_state *st, const bz_selfplay_endgame_state *eg,
                            const bz_selfplay_resign_state *rs, const bz_selfplay_cap_state *cs,
                            const bz_tree_pools *pools, uint8_t *action_out, bz_stream_t stream) {
    int rc = check_state(st);
    if (rc != BZ_OK) return rc;
    if (eg && (rc = check_endgame(st, eg)) != BZ_OK) return rc;
    if (rs && (rc = check_resign(eg, rs)) != BZ_OK) return rc;
    rc = check_cap(st, eg, cs);
    if (rc != BZ_OK) return rc;
    if (!pools || pools->game != BZ_GAME_REVERSI || pools->n_trees != cs->n_trees || pools->board_size != st->board_size ||
        !pools->root_meta || !pools->arena)
        return BZ_ERR_ARG;
    if (st->n_games == 0) return BZ_OK;
    const unsigned grid = (st->n_games + kWarpsPerCta - 1) / kWarpsPerCta;
    const uint64_t cells = cell_mask(st->board_size);
    const bz_selfplay_endgame_state no_eg = {};
    const bz_selfplay_resign_state no_rs = {};
    const cudaStream_t s = as_stream(stream);
    if (eg && rs) {
        selfplay_advance_cap_kernel<true, true><<<grid, kThreads, 0, s>>>(*st, *pools, action_out, cells, *eg, *rs, *cs);
    } else if (eg) {
        selfplay_advance_cap_kernel<true, false><<<grid, kThreads, 0, s>>>(*st, *pools, action_out, cells, *eg, no_rs, *cs);
    } else if (rs) {
        selfplay_advance_cap_kernel<false, true><<<grid, kThreads, 0, s>>>(*st, *pools, action_out, cells, no_eg, *rs, *cs);
    } else {
        selfplay_advance_cap_kernel<false, false><<<grid, kThreads, 0, s>>>(*st, *pools, action_out, cells, no_eg, no_rs,
                                                                           *cs);
    }
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
        *st, *pools, cell_mask(st->board_size), 0ull, nullptr);
    return launch_rc();
}

int bz_tournament_minimax(const bz_tournament_state *st, const int32_t *entrant_depth, void *workspace, uint8_t *action,
                          int64_t *nodes_total, bz_stream_t stream) {
    int rc = check_tournament(st);
    if (rc != BZ_OK) return rc;
    if (!entrant_depth || !workspace || !action) return BZ_ERR_ARG;
    if (!aligned16(workspace)) return BZ_ERR_UNALIGNED;
    MinimaxRoots R = {};
    R.me = st->match.root_me;
    R.opp = st->match.root_opp;
    R.n = st->match.n_trees;
    R.game_of_tree = st->match.game_of_tree;
    R.pair_entrant = st->match.pair_net;
    R.key_base = 2 * st->match.first_pair_id;
    for (int e = 0; e < BZ_MAX_ENTRANTS; ++e) R.entrant_depth[e] = kMinimaxNotSearched;
    for (int e = 0; e < st->n_entrants; ++e) {
        const int d = entrant_depth[e];
        if (d < -1 || d > BZ_MINIMAX_MAX_DEPTH) return BZ_ERR_ARG;
        if (d >= 0) R.entrant_depth[e] = (uint8_t)d;
    }
    return minimax_launch(R, st->match.seed, st->match.board_size, workspace, action, nullptr, nullptr, nodes_total,
                          as_stream(stream));
}

int bz_tournament_advance(const bz_tournament_state *st, const bz_tree_pools *pools, const int32_t *entrant_depth,
                          const uint8_t *action, bz_stream_t stream) {
    int rc = check_tournament(st);
    if (rc != BZ_OK) return rc;
    if (!entrant_depth || !action) return BZ_ERR_ARG;
    uint64_t bits = 0;
    bool nets = false;
    for (int e = 0; e < st->n_entrants; ++e) {
        const int d = entrant_depth[e];
        if (d < -1 || d > BZ_MINIMAX_MAX_DEPTH) return BZ_ERR_ARG;
        if (d >= 0) bits |= 1ull << e;
        else nets = true;
    }
    bz_tree_pools P = {};
    if (nets || pools) {
        if (!pools || pools->game != BZ_GAME_REVERSI || pools->n_trees != st->match.n_trees ||
            pools->board_size != st->match.board_size || !pools->root_meta || !pools->arena)
            return BZ_ERR_ARG;
        P = *pools;
    }
    if (st->match.n_games == 0) return BZ_OK;
    match_advance_kernel<<<(st->match.n_games + kWarpsPerCta - 1) / kWarpsPerCta, kThreads, 0, as_stream(stream)>>>(
        st->match, P, cell_mask(st->match.board_size), bits, action);
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
