// Depth-limited minimax for sm_100a: the reference's OptimalPlayer.get_move (src/reversi/players/reversi_players.py:35-77)
// for thousands of roots at once.  Definition: oracle/minimax_ref.py; semantics: include/betazero_b200.h (bz_minimax_moves).
//
// Shape: the search is split at the root.  Every (root, root move) is one work item, searched by one thread with
// alpha-beta in row-major order and the full window, so each child's value is exact; the root then takes the first
// maximum, as the reference's strict ">" does.  Node counts of the items differ by orders of magnitude, so a persistent
// grid hands the items out from an atomic counter, and a thread takes its next item as soon as its search ends (a step of
// the search loop is either a descent or a return, whichever item the lane holds).  Four launches:
//   prep   (thread per root): legal moves, the answer of roots that need no search, the item count of the others
//   scan   (one CTA): item offsets
//   search (persistent): the items
//   finish (thread per root): first maximum, or the Philox move; node totals
// The whole-board shape (one item per root, the window passed on between root moves: fewer nodes) was 3.0 - 4.1x slower
// at depths 3 - 6 on 4096 mid-game roots (DESIGN.md section 7).
//
// The endgame solver (bz_endgame_solve; definition: oracle/endgame_ref.py) searches to the end of the game with
// passes, split at two plies; it has its own prep and finish kernels and shares the workspace layout, the scan and the
// item search with minimax.  Its win/draw/loss form (bz_endgame_solve_wld) is the same kernels instantiated with kWld:
// a null window and fastest-first move ordering.  Self-play's endgame queue (selfplay.cu) runs the same kernels with
// its root count read from device memory (endgame_launch_live).
//
// The item search (search_kernel) is one negamax loop for both solvers, with a struct per solver for what differs.
// Minimax in negamax form visits the reference's nodes: its value at depth d is (-1)^d times the value for the mover, a
// min node's beta update is the negamax alpha update on the negated window, and the initial best differs only at a node
// without children, which the node rule ends first.
#include "bitboard.cuh"
#include "common.cuh"
#include "minimax.cuh"

namespace bz {
namespace {

constexpr int kD0 = 1;  // absolute depth of a work item's first node: a root move's child
constexpr int kInf = 127;      // the value of +-inf
constexpr int kWindow = 128;   // the full window (-128, 128) holds every value, +-inf included
constexpr int kSlots = 64;     // per root in the workspace's value array: more than any position's move count
constexpr int kSkip = -1;      // root not searched
constexpr int kSearchThreads = 128;

struct Workspace {
    unsigned *counter;   // [0] next item, [1] items
    unsigned *offset;    // [n + 1]: first item of each root
    unsigned long long *nodes;  // [n]
    int8_t *vals;        // [n * kSlots]: value of each root move
};

__host__ __device__ inline int64_t align16(int64_t b) { return (b + 15) & ~(int64_t)15; }

Workspace carve(void *base, int64_t n) {
    char *p = static_cast<char *>(base);
    Workspace w;
    w.counter = reinterpret_cast<unsigned *>(p);
    p += 16;
    w.offset = reinterpret_cast<unsigned *>(p);
    p += align16(4 * (n + 1));
    w.nodes = reinterpret_cast<unsigned long long *>(p);
    p += align16(8 * n);
    w.vals = reinterpret_cast<int8_t *>(p);
    return w;
}

// depth of root i (0 .. BZ_MINIMAX_MAX_DEPTH), or kSkip; its game key
__device__ __forceinline__ int root_depth(const MinimaxRoots &R, int64_t i, uint64_t &key) {
    if (R.depth) {
        const int d = R.depth[i];
        BZ_CHECK(d <= BZ_MINIMAX_MAX_DEPTH, 60);  // depth out of range: the root is not searched
        key = R.key[i];
        return d <= BZ_MINIMAX_MAX_DEPTH ? d : kSkip;
    }
    const int g = R.game_of_tree[i];
    if (g < 0) return kSkip;  // padding
    const int e = R.pair_entrant[i / BZ_MATCH_TREES_PER_PAIR];
    BZ_CHECK(e < BZ_MAX_ENTRANTS, 61);  // entrant id
    if (e >= BZ_MAX_ENTRANTS) return kSkip;
    const int d = R.entrant_depth[e];
    key = (uint64_t)(R.key_base + g);
    return d <= BZ_MINIMAX_MAX_DEPTH ? d : kSkip;  // a net entrant's tree
}

// the reference's random.choice(moves) (reversi_players.py:42-43), reproducibly: Philox keyed by 2^32 + the game key,
// counter = discs on the board
__device__ __forceinline__ unsigned random_move(uint64_t seed, uint64_t key, uint64_t me, uint64_t opp, uint64_t m) {
    return pick_move(m, philox_u32(seed, (1ull << 32) + key, (uint32_t)__popcll(me | opp)));
}

__global__ void __launch_bounds__(256) minimax_prep_kernel(const MinimaxRoots R, uint64_t seed, uint64_t cells, Workspace W,
                                                           uint8_t *action, int8_t *value) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= R.n) return;
    uint64_t key = 0;
    const int d = root_depth(R, i, key);
    unsigned cnt = 0;
    if (d == kSkip) {
        action[i] = 255u;
        if (value) value[i] = 0;
        W.nodes[i] = 0;
    } else {
        const uint64_t me = R.me[i], opp = R.opp[i];
        const uint64_t m = legal_mask(me, opp, cells);
        const int ev = __popcll(me) - __popcll(opp);
        W.nodes[i] = 1;
        if (m == 0) {  // the game is over (255), or the player must pass (64): the reference searches nothing here
            const bool over = legal_mask(opp, me, cells) == 0;
            action[i] = over ? 255u : 64u;
            if (value) value[i] = (int8_t)((d == 0 || over) ? ev : -kInf);
        } else if (d == 0) {
            action[i] = (uint8_t)random_move(seed, key, me, opp, m);
            if (value) value[i] = (int8_t)ev;
        } else {
            cnt = (unsigned)__popcll(m);
        }
    }
    W.offset[i] = cnt;
}

// exclusive scan of the item counts in place; offset[n] = items; resets the item counter
__global__ void __launch_bounds__(1024) minimax_scan_kernel(Workspace W, int64_t n) {
    __shared__ unsigned warp_sum[32];
    __shared__ unsigned carry_s;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    unsigned carry = 0;
    for (int64_t base = 0; base < n; base += 1024) {
        const int64_t i = base + tid;
        const unsigned v = i < n ? W.offset[i] : 0u;
        unsigned incl = v;
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned up = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += up;
        }
        if (lane == 31) warp_sum[w] = incl;
        __syncthreads();
        if (w == 0) {
            const unsigned s = warp_sum[lane];
            unsigned si = s;
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned up = __shfl_up_sync(0xFFFFFFFFu, si, d);
                if (lane >= d) si += up;
            }
            warp_sum[lane] = si - s;
            if (lane == 31) carry_s = si;
        }
        __syncthreads();
        if (i < n) W.offset[i] = carry + warp_sum[w] + incl - v;
        carry += carry_s;
        __syncthreads();
    }
    if (tid == 0) {
        W.offset[n] = carry;
        W.counter[0] = 0;
        W.counter[1] = carry;
    }
}

// the root of item i: the largest r with offset[r] <= i (roots without items share their successor's offset)
__device__ __forceinline__ int64_t item_root(const unsigned *offset, int64_t n, unsigned i) {
    int64_t lo = 0, hi = n - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (offset[mid] <= i) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// the persistent hand-out: the next item i from the atomic counter and its root; false when every item is taken.  The
// item's index among its root's items is i - offset[root].
__device__ __forceinline__ bool take_item(const Workspace &W, int64_t n, unsigned total, int64_t &root, unsigned &i) {
    i = atomicAdd(&W.counter[0], 1u);
    if (i >= total) return false;
    root = item_root(W.offset, n, i);
    BZ_CHECK(root >= 0 && root < n && W.offset[root] <= i && i < W.offset[root + 1], 62);  // item -> root
    return true;
}

__global__ void __launch_bounds__(256) minimax_finish_kernel(const MinimaxRoots R, uint64_t seed, uint64_t cells, Workspace W,
                                                             uint8_t *action, int8_t *value, int64_t *nodes,
                                                             int64_t *nodes_total) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned long long nd = 0;
    if (i < R.n) {
        nd = W.nodes[i];
        const unsigned cnt = W.offset[i + 1] - W.offset[i];
        if (cnt) {
            uint64_t key = 0;
            root_depth(R, i, key);
            const uint64_t me = R.me[i], opp = R.opp[i], m = legal_mask(me, opp, cells);
            int best = -kInf, bj = -1;
            BZ_CHECK(cnt <= (unsigned)kSlots, 66);  // value slots
            for (unsigned j = 0; j < cnt; ++j) {
                const int x = W.vals[i * kSlots + j];
                if (x > best) {  // the first maximum (reversi_players.py:56-58)
                    best = x;
                    bj = (int)j;
                }
            }
            action[i] = (uint8_t)(bj >= 0 ? kth_bit(m, bj) : random_move(seed, key, me, opp, m));
            if (value) value[i] = (int8_t)best;
        }
        if (nodes) nodes[i] = (int64_t)nd;
    }
    if (nodes_total) {
        for (int d = 16; d; d >>= 1) nd += __shfl_xor_sync(0xFFFFFFFFu, nd, d);
        if ((threadIdx.x & 31) == 0 && nd) atomicAdd(reinterpret_cast<unsigned long long *>(nodes_total), nd);
    }
}

// ---- the endgame solver (bz_endgame_solve) --------------------------------------------------------------------------
// Exact negamax to the end of the game, passes included.  Shape: split at two plies.  Every (root, root move, reply) is
// one work item, and so is a root move whose child must pass or is finished; one thread searches it with alpha-beta in
// row-major order and the full window, so the item's value is exact.  move_value[a] is the minimum over a's items
// (atomicMin into the workspace), and the finish kernel takes the first maximum.  A root that must pass has the pass as
// its one move.  Workspace, scan and the item search are those of minimax.
//
// The win/draw/loss solve (kWld; bz_endgame_solve_wld) runs the same items with the null window (-1, 1): fail-soft, an
// item's value v >= 1 is a win, v <= -1 a loss and 0 an exact draw, so clamped to [-1, 1] it is the sign of the exact
// value, and so is the minimum over a move's replies.  At every node with at least kOrderEmpties empties it tries the
// moves fastest first: fewest legal replies for the opponent first, ties in cell order.  Below that it keeps the
// row-major descent, where ordering costs more than the cutoffs it finds.  Items share no bounds, so an item's node
// count depends on its root alone.
constexpr int kSolveLevels = BZ_SOLVE_MAX_EMPTIES + 1;  // a level per disc placed; a pass stays on its level
constexpr int kMoveSlots = 65;  // move values per root: 64 cells and the pass
constexpr int kUnset = 127;     // a move value no item has bounded yet
constexpr int64_t kSolveChunk = (int64_t)1 << 22;  // roots per set of launches: at most 380 items each fit 32-bit offsets
#ifndef BZ_SOLVE_ORDER_EMPTIES
#define BZ_SOLVE_ORDER_EMPTIES 6  // the fastest of T = 6, 8, 10, 12 and none at 12 and 14 empties (profiles/README.md)
#endif
constexpr int kOrderEmpties = BZ_SOLVE_ORDER_EMPTIES;
// an item's first node has at most BZ_SOLVE_MAX_EMPTIES - 1 empties, so levels below this hold every ordered node
constexpr int kOrderLevels = BZ_SOLVE_MAX_EMPTIES - kOrderEmpties > 0 ? BZ_SOLVE_MAX_EMPTIES - kOrderEmpties : 1;
constexpr int kOrderMoves = BZ_SOLVE_MAX_EMPTIES;  // a move per empty square at most

// the k-th move of a root whose legal moves are m (the pass when m == 0): its action and child, mover-relative
__device__ __forceinline__ unsigned root_move(uint64_t me, uint64_t opp, uint64_t m, int k, uint64_t &cme, uint64_t &copp) {
    const unsigned a = m ? kth_bit(m, k) : 64u;
    cme = me;
    copp = opp;
    apply_legal(cme, copp, a);
    return a;
}

__device__ __forceinline__ int solve_empties(uint64_t me, uint64_t opp, uint64_t cells) {
    return __popcll(cells) - __popcll((me | opp) & cells);
}

// fastest first: the moves m of (me, opp) as keys (the opponent's legal-move count after the move) << 6 | cell, in
// ascending order (ties in cell order); the ordering's positions are not counted as nodes
__device__ __forceinline__ void order_moves(uint64_t me, uint64_t opp, uint64_t m, uint64_t cells, uint16_t *keys) {
    for (int n = 0; m; m &= m - 1, ++n) {
        const unsigned a = (unsigned)(__ffsll((long long)m) - 1);
        uint64_t cme = me, copp = opp;
        apply_legal(cme, copp, a);
        const unsigned key = (unsigned)__popcll(legal_mask(cme, copp, cells)) << 6 | a;
        int j = n;
        for (; j > 0 && keys[j - 1] > key; --j) keys[j] = keys[j - 1];
        keys[j] = (uint16_t)key;
    }
}

// kLive: the roots are [0, *live) of n (the self-play endgame queue: launch shapes depend on n only); the others get
// no items.  kWld: a finished root's value is the sign of its disc difference.
template <bool kLive, bool kWld>
__global__ void __launch_bounds__(256) endgame_prep_kernel(const uint64_t *me_, const uint64_t *opp_, int64_t n,
                                                           uint64_t cells, Workspace W, uint8_t *action, int8_t *value,
                                                           const int32_t *live) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (kLive && i >= *live) {
        W.nodes[i] = 0;
        W.offset[i] = 0;
        return;
    }
    int *mv = reinterpret_cast<int *>(W.vals) + i * kMoveSlots;
    for (int j = 0; j < kMoveSlots; ++j) mv[j] = kUnset;
    const uint64_t me = me_[i], opp = opp_[i];
    unsigned cnt = 0;
    unsigned long long nd = 0;
    const bool fits = solve_empties(me, opp, cells) <= BZ_SOLVE_MAX_EMPTIES;
    BZ_CHECK(fits, 70);  // too many empties: the root is not searched
    const uint64_t m = legal_mask(me, opp, cells);
    if (!fits || (m == 0 && legal_mask(opp, me, cells) == 0)) {  // not searched, or the game is over
        action[i] = 255u;
        const int d = __popcll(me) - __popcll(opp);
        value[i] = (int8_t)(fits ? (kWld ? (d > 0) - (d < 0) : d) : 0);
        nd = fits;
    } else {
        const int moves = m ? __popcll(m) : 1;
        nd = 1;
        for (int k = 0; k < moves; ++k) {
            uint64_t cme, copp;
            root_move(me, opp, m, k, cme, copp);
            const int c = __popcll(legal_mask(cme, copp, cells));
            cnt += c ? c : 1;
            ++nd;  // the child, entered here for its items
        }
    }
    W.nodes[i] = nd;
    W.offset[i] = cnt;
}

// ---- the item search of both solvers --------------------------------------------------------------------------------
// Fail-soft alpha-beta negamax of one item per thread from the item's first node.  S supplies what differs between the
// solvers: kLevels (the stack depth), kOrdered (fastest first at nodes with at least kOrderEmpties empties), roots(),
// first() (the item's first node and window (-w, w), or false and the value of an item whose game is over: the prep
// kernel entered its node), node() (the node rule: kLeaf and the value for the node's mover, kInner and the moves, or
// kPass and the opponent's moves) and store() (the value of the item's first node, for its mover).
enum NodeKind { kInner, kLeaf, kPass };

template <class S>
__global__ void __launch_bounds__(kSearchThreads) search_kernel(const S s, Workspace W) {
    const unsigned total = W.counter[1];
    // the stack of the item's search: level k holds the node k plies below the item's first node; a node whose mover
    // must pass is held as the position after the pass, with bit k of `passed` set and its window negated
    uint64_t s_me[S::kLevels], s_opp[S::kLevels], s_rem[S::kLevels];
    int s_best[S::kLevels], s_alpha[S::kLevels], s_beta[S::kLevels];
    // S::kOrdered: a level with bit k of `ordered` set descends in the order of s_order[k] from s_cur[k] (order_moves)
    uint16_t s_order[kOrderLevels][kOrderMoves];
    uint8_t s_cur[kOrderLevels];
    unsigned ordered = 0;
    unsigned passed = 0;
    int k = -1;  // level of the node being searched; -1: no item
    int v = 0;
    int64_t root = 0;
    unsigned slot = 0;
    typename S::Item it;
    unsigned long long nodes = 0;
    bool leaf = false;

    // enter the node (me, opp) at level k with the window (alpha, beta): a leaf sets v, any other node its moves
    auto enter = [&](uint64_t me, uint64_t opp, int alpha, int beta) {
        ++nodes;
        passed &= ~(1u << k);
        uint64_t m = 0;
        const NodeKind kind = s.node(me, opp, k, it, m, v);
        if (kind == kLeaf) {
            leaf = true;
            return;
        }
        if (kind == kPass) {
            ++nodes;  // the position after the pass
            passed |= 1u << k;
            const uint64_t t = me;
            me = opp;
            opp = t;
            const int a = alpha;
            alpha = -beta;
            beta = -a;
        }
        s_me[k] = me;
        s_opp[k] = opp;
        s_rem[k] = m;
        s_best[k] = -kWindow;
        s_alpha[k] = alpha;
        s_beta[k] = beta;
        if constexpr (S::kOrdered) {
            ordered &= ~(1u << k);
            if (k < kOrderLevels && solve_empties(me, opp, s.cells) >= kOrderEmpties) {
                order_moves(me, opp, m, s.cells, s_order[k]);
                s_cur[k] = 0;
                ordered |= 1u << k;
            }
        }
        leaf = false;
    };

    while (true) {
        if (k < 0) {
            if (!take_item(W, s.roots(), total, root, slot)) break;
            slot -= W.offset[root];
            nodes = 0;
            k = 0;
            uint64_t me = 0, opp = 0;
            int w = 0;
            if (s.first(root, slot, it, me, opp, w, v)) enter(me, opp, -w, w);
            else leaf = true;
        } else if (!leaf) {  // descend into the next move of level k: row-major, or in the level's order
            const uint64_t rem = s_rem[k];
            uint64_t x = rem & (0ull - rem);
            if constexpr (S::kOrdered) {
                if ((ordered >> k) & 1u) x = 1ull << (s_order[k][s_cur[k]++] & 63u);
            }
            s_rem[k] = rem ^ x;
            uint64_t me = s_me[k], opp = s_opp[k];
            apply_legal(me, opp, (unsigned)(__ffsll((long long)x) - 1));
            BZ_CHECK(k + 1 < S::kLevels, 64);  // stack level
            const int alpha = s_alpha[k], beta = s_beta[k];
            ++k;
            enter(me, opp, -beta, -alpha);
        }
        if (!leaf) continue;
        // return v, the value of level k's node for its mover, to the parents until one has a move left to search
        while (true) {
            if (k == 0) {
                s.store(W, root, slot, it, v);
                if (nodes) atomicAdd(&W.nodes[root], nodes);
                k = -1;
                break;
            }
            --k;
            const int x = -v;
            int best = s_best[k];
            if (x > best) best = x;
            s_best[k] = best;
            if (best > s_alpha[k]) s_alpha[k] = best;
            if (s_alpha[k] >= s_beta[k] || s_rem[k] == 0) {
                v = (passed >> k) & 1u ? -best : best;
                continue;
            }
            leaf = false;
            break;
        }
    }
}

// minimax: the item of root move `slot` is that move's child, the opponent's node, searched to the root's depth
struct MinimaxItems {
    static constexpr int kLevels = BZ_MINIMAX_MAX_DEPTH + 1;
    static constexpr bool kOrdered = false;
    struct Item { int depth; };
    MinimaxRoots R;
    uint64_t cells;

    __device__ __forceinline__ int64_t roots() const { return R.n; }

    __device__ __forceinline__ bool first(int64_t root, unsigned slot, Item &it, uint64_t &me, uint64_t &opp, int &w,
                                          int &) const {
        uint64_t key;
        it.depth = root_depth(R, root, key);
        me = R.me[root];
        opp = R.opp[root];
        BZ_CHECK(slot < (unsigned)kSlots, 63);  // value slot
        apply_legal(me, opp, kth_bit(legal_mask(me, opp, cells), (int)slot));
        w = kWindow;
        return true;
    }

    // at the depth limit the disc difference; without a move the disc difference if the game is over, otherwise -inf:
    // the reference's search does not pass, its loop over no moves returns the initial -inf (for the mover)
    __device__ __forceinline__ NodeKind node(uint64_t me, uint64_t opp, int k, const Item &it, uint64_t &m,
                                             int &v) const {
        v = __popcll(me) - __popcll(opp);
        if (kD0 + k >= it.depth) return kLeaf;
        m = legal_mask(me, opp, cells);
        if (m) return kInner;
        if (legal_mask(opp, me, cells)) v = -kInf;
        return kLeaf;
    }

    __device__ __forceinline__ void store(const Workspace &W, int64_t root, unsigned slot, const Item &, int v) const {
        BZ_CHECK(root * kSlots + slot < R.n * kSlots, 65);  // value slot
        W.vals[root * kSlots + slot] = (int8_t)-v;  // the root mover's view of the opponent's node
    }
};

// the endgame solver: the item is a (root move, reply) decoded from its index, or a root move whose child must pass or
// is finished; kWld: the null window and move ordering
template <bool kWld>
struct EndgameItems {
    static constexpr int kLevels = kSolveLevels;
    static constexpr bool kOrdered = kWld;
    struct Item { unsigned move; };  // the root move
    const uint64_t *root_me, *root_opp;
    int64_t n;
    uint64_t cells;

    __device__ __forceinline__ int64_t roots() const { return n; }

    __device__ __forceinline__ bool first(int64_t root, unsigned slot, Item &it, uint64_t &me, uint64_t &opp, int &w,
                                          int &v) const {
        const uint64_t rme = root_me[root], ropp = root_opp[root], m = legal_mask(rme, ropp, cells);
        const int moves = m ? __popcll(m) : 1;
        uint64_t cme = 0, copp = 0, cm = 0;
        unsigned r = slot;
        for (int j = 0; j < moves; ++j) {  // the root move of the item, and the reply's index r
            it.move = root_move(rme, ropp, m, j, cme, copp);
            cm = legal_mask(cme, copp, cells);
            const unsigned c = cm ? (unsigned)__popcll(cm) : 1u;
            if (r < c) break;
            r -= c;
        }
        BZ_CHECK(r < (cm ? (unsigned)__popcll(cm) : 1u), 71);  // reply
        if (!cm && !legal_mask(copp, cme, cells)) {
            v = __popcll(copp) - __popcll(cme);  // the child's game is over: the root mover's count
            return false;
        }
        apply_legal(cme, copp, cm ? kth_bit(cm, (int)r) : 64u);  // the child passes: the item is the position after it
        me = cme;
        opp = copp;
        w = kWld ? 1 : kWindow;  // the null window, or the full one
        return true;
    }

    // a finished game: the disc difference, empty squares to nobody; no move: a pass
    __device__ __forceinline__ NodeKind node(uint64_t me, uint64_t opp, int, const Item &, uint64_t &m, int &v) const {
        m = legal_mask(me, opp, cells);
        if (m) return kInner;
        m = legal_mask(opp, me, cells);
        if (m) return kPass;
        v = __popcll(me) - __popcll(opp);
        return kLeaf;
    }

    // the item's first node belongs to the root's mover: a move's value is its items' minimum
    __device__ __forceinline__ void store(const Workspace &W, int64_t root, unsigned, const Item &it, int v) const {
        BZ_CHECK(root * kMoveSlots + it.move < n * kMoveSlots, 73);  // move value slot
        if constexpr (kWld) v = v > 1 ? 1 : (v < -1 ? -1 : v);  // a bound beyond the null window: its sign
        atomicMin(reinterpret_cast<int *>(W.vals) + root * kMoveSlots + it.move, v);
    }
};

template <bool kLive>
__global__ void __launch_bounds__(256) endgame_finish_kernel(const uint64_t *me_, const uint64_t *opp_, int64_t n,
                                                             uint64_t cells, Workspace W, uint8_t *action, int8_t *value,
                                                             int8_t *move_value, int64_t *nodes, const int32_t *live) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n || (kLive && i >= *live)) return;
    const int *mv = reinterpret_cast<const int *>(W.vals) + i * kMoveSlots;
    int8_t *out = move_value + i * kMoveSlots;
    if (W.offset[i + 1] != W.offset[i]) {  // searched
        const uint64_t m = legal_mask(me_[i], opp_[i], cells);
        int best = -kWindow, bj = 255;
        for (int j = 0; j < kMoveSlots; ++j) {
            const bool legal = j < 64 ? ((m >> j) & 1) != 0 : m == 0;
            int x = -kWindow;
            if (legal) {
                x = mv[j];
                BZ_CHECK(x != kUnset, 74);  // a move without a value
                if (x > best) {  // the first maximum: the reference's strict ">"
                    best = x;
                    bj = j;
                }
            }
            out[j] = (int8_t)x;
        }
        action[i] = (uint8_t)bj;
        value[i] = (int8_t)best;
    } else {
        for (int j = 0; j < kMoveSlots; ++j) out[j] = (int8_t)-kWindow;
    }
    if (nodes) nodes[i] = (int64_t)W.nodes[i];
}

}  // namespace

int64_t minimax_workspace_bytes(int64_t n) {
    if (n < 0) return 0;
    return 16 + align16(4 * (n + 1)) + align16(8 * n) + align16((int64_t)kSlots * n);
}

int minimax_launch(const MinimaxRoots &R, uint64_t seed, int size, void *workspace, uint8_t *action, int8_t *value,
                   int64_t *nodes, int64_t *nodes_total, cudaStream_t stream) {
    if (R.n == 0) return BZ_OK;
    const uint64_t cells = cell_mask(size);
    const Workspace W = carve(workspace, R.n);
    const unsigned blocks = (unsigned)((R.n + 255) / 256);
    minimax_prep_kernel<<<blocks, 256, 0, stream>>>(R, seed, cells, W, action, value);
    minimax_scan_kernel<<<1, 1024, 0, stream>>>(W, R.n);
    search_kernel<<<persistent_grid(R.n * 32, kSearchThreads, 8), kSearchThreads, 0, stream>>>(MinimaxItems{R, cells}, W);
    minimax_finish_kernel<<<blocks, 256, 0, stream>>>(R, seed, cells, W, action, value, nodes, nodes_total);
    return launch_rc();
}

// the minimax layout with an int32 move value per (root, action) in place of the int8 values of the root moves
int64_t endgame_workspace_bytes(int64_t n) {
    if (n < 0) return 0;
    const int64_t c = n < kSolveChunk ? n : kSolveChunk;
    return 16 + align16(4 * (c + 1)) + align16(8 * c) + align16(4 * kMoveSlots * c);
}

// the solver's four launches over n <= kSolveChunk roots (live: the roots [0, *live), see endgame_prep_kernel)
template <bool kLive, bool kWld>
void endgame_kernels(const uint64_t *me, const uint64_t *opp, int64_t n, const int32_t *live, uint64_t cells,
                     const Workspace &W, uint8_t *action, int8_t *value, int8_t *move_value, int64_t *nodes,
                     cudaStream_t stream) {
    const unsigned blocks = (unsigned)((n + 255) / 256);
    endgame_prep_kernel<kLive, kWld><<<blocks, 256, 0, stream>>>(me, opp, n, cells, W, action, value, live);
    minimax_scan_kernel<<<1, 1024, 0, stream>>>(W, n);  // the roots past *live have no items: no item maps to them
    search_kernel<<<persistent_grid(n * 64, kSearchThreads, 8), kSearchThreads, 0, stream>>>(
        EndgameItems<kWld>{me, opp, n, cells}, W);
    endgame_finish_kernel<kLive><<<blocks, 256, 0, stream>>>(me, opp, n, cells, W, action, value, move_value, nodes,
                                                             live);
}

int endgame_launch(const uint64_t *me, const uint64_t *opp, int64_t n, int size, void *workspace, uint8_t *action,
                   int8_t *value, int8_t *move_value, int64_t *nodes, bool wld, cudaStream_t stream) {
    const uint64_t cells = cell_mask(size);
    for (int64_t b = 0; b < n; b += kSolveChunk) {  // stream order makes the chunks' reuse of the workspace safe
        const int64_t c = n - b < kSolveChunk ? n - b : kSolveChunk;
        const Workspace W = carve(workspace, c);
        (wld ? endgame_kernels<false, true> : endgame_kernels<false, false>)(
            me + b, opp + b, c, nullptr, cells, W, action + b, value + b, move_value + b * kMoveSlots,
            nodes ? nodes + b : nullptr, stream);
        const int rc = launch_rc();
        if (rc != BZ_OK) return rc;
    }
    return BZ_OK;
}

int endgame_launch_live(const uint64_t *me, const uint64_t *opp, int64_t n, const int32_t *live, int size, void *workspace,
                        uint8_t *action, int8_t *value, int8_t *move_value, bool wld, cudaStream_t stream) {
    if (n <= 0 || n > kSolveChunk) return BZ_ERR_ARG;
    const Workspace W = carve(workspace, n);
    (wld ? endgame_kernels<true, true> : endgame_kernels<true, false>)(me, opp, n, live, cell_mask(size), W, action,
                                                                       value, move_value, nullptr, stream);
    return launch_rc();
}

}  // namespace bz

using namespace bz;

extern "C" {

int64_t bz_minimax_workspace_bytes(int64_t n) { return minimax_workspace_bytes(n); }

int bz_minimax_moves(const uint64_t *me, const uint64_t *opp, const uint8_t *depth, const uint64_t *key, uint64_t seed,
                     int64_t n, int size, void *workspace, uint8_t *action, int8_t *value, int64_t *nodes,
                     bz_stream_t stream) {
    if (!(size == 4 || size == 6 || size == 8) || n < 0 || n >= (int64_t)1 << 25) return BZ_ERR_ARG;
    if (n == 0) return BZ_OK;
    if (!me || !opp || !depth || !key || !workspace || !action || !value) return BZ_ERR_ARG;
    if (!aligned16(workspace)) return BZ_ERR_UNALIGNED;
    MinimaxRoots R = {};
    R.me = me;
    R.opp = opp;
    R.n = n;
    R.depth = depth;
    R.key = key;
    return minimax_launch(R, seed, size, workspace, action, value, nodes, nullptr, as_stream(stream));
}

int64_t bz_endgame_workspace_bytes(int64_t n) { return endgame_workspace_bytes(n); }

static int endgame_solve(const uint64_t *me, const uint64_t *opp, int64_t n, int size, void *workspace, uint8_t *action,
                         int8_t *value, int8_t *move_value, int64_t *nodes, bool wld, bz_stream_t stream) {
    if (!(size == 4 || size == 6 || size == 8) || n < 0 || n >= (int64_t)1 << 25) return BZ_ERR_ARG;
    if (n == 0) return BZ_OK;
    if (!me || !opp || !workspace || !action || !value || !move_value) return BZ_ERR_ARG;
    if (!aligned16(workspace)) return BZ_ERR_UNALIGNED;
    return endgame_launch(me, opp, n, size, workspace, action, value, move_value, nodes, wld, as_stream(stream));
}

int bz_endgame_solve(const uint64_t *me, const uint64_t *opp, int64_t n, int size, void *workspace, uint8_t *action,
                     int8_t *value, int8_t *move_value, int64_t *nodes, bz_stream_t stream) {
    return endgame_solve(me, opp, n, size, workspace, action, value, move_value, nodes, false, stream);
}

int bz_endgame_solve_wld(const uint64_t *me, const uint64_t *opp, int64_t n, int size, void *workspace, uint8_t *action,
                         int8_t *value, int8_t *move_value, int64_t *nodes, bz_stream_t stream) {
    return endgame_solve(me, opp, n, size, workspace, action, value, move_value, nodes, true, stream);
}

}  // extern "C"

#ifdef BZ_BOUNDS_CHECK
// debug builds: [code of the first failed check, block, thread, violations] of the minimax kernels; clears the record
extern "C" int bz_debug_checks_minimax(int *host_out) {
    int rc = bz::cuda_rc(cudaMemcpyFromSymbol(host_out, bz::g_bz_check, sizeof(int) * 4));
    if (rc) return rc;
    const int zero[4] = {0, 0, 0, 0};
    return bz::cuda_rc(cudaMemcpyToSymbol(bz::g_bz_check, zero, sizeof(zero)));
}
#endif
