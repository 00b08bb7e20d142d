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
#include "bitboard.cuh"
#include "common.cuh"
#include "minimax.cuh"

namespace bz {
namespace {

constexpr int kD0 = 1;  // absolute depth of a work item's first node: a root move's child
constexpr int kLevels = BZ_MINIMAX_MAX_DEPTH + 1;
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

__device__ __forceinline__ unsigned kth_bit(uint64_t m, int k) {
    for (; k > 0; --k) m &= m - 1;
    return (unsigned)(__ffsll((long long)m) - 1);
}

// the reference's random.choice(moves) (reversi_players.py:42-43), reproducibly: Philox keyed by 2^32 + the game key,
// counter = discs on the board; the k-th legal move in ascending cell order, k = floor(u * moves / 2^32)
__device__ __forceinline__ unsigned random_move(uint64_t seed, uint64_t key, uint64_t me, uint64_t opp, uint64_t m) {
    const uint32_t u = philox_u32(seed, (1ull << 32) + key, (uint32_t)__popcll(me | opp));
    return kth_bit(m, (int)(((uint64_t)u * (uint64_t)__popcll(m)) >> 32));
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

__global__ void __launch_bounds__(kSearchThreads) minimax_search_kernel(const MinimaxRoots R, uint64_t cells, Workspace W) {
    const unsigned total = W.counter[1];
    // the stack of the item's search: level k holds the node at absolute depth kD0 + k
    uint64_t s_me[kLevels], s_opp[kLevels], s_rem[kLevels];
    int s_best[kLevels], s_alpha[kLevels], s_beta[kLevels];
    int k = -1;  // level of the node being searched; -1: no item
    int depth = 0, v = 0;
    int64_t root = 0;
    unsigned slot = 0, nodes = 0;
    bool leaf = false;

    // enter the node (me, opp) at level k: a leaf sets v, an inner node its moves and initial best
    auto enter = [&](uint64_t me, uint64_t opp) {
        const int d = kD0 + k;
        const bool maxing = (d & 1) == 0;
        s_me[k] = me;
        s_opp[k] = opp;
        const int ev = maxing ? __popcll(me) - __popcll(opp) : __popcll(opp) - __popcll(me);
        if (d >= depth) {
            v = ev;
            leaf = true;
            return;
        }
        const uint64_t m = legal_mask(me, opp, cells);
        if (m == 0) {  // game over: evaluate; otherwise the loop over no moves returns the initial -inf / +inf
            v = legal_mask(opp, me, cells) == 0 ? ev : (maxing ? -kInf : kInf);
            leaf = true;
            return;
        }
        s_rem[k] = m;
        s_best[k] = maxing ? -kInf : kInf;
        leaf = false;
    };

    while (true) {
        if (k < 0) {
            const unsigned i = atomicAdd(&W.counter[0], 1u);
            if (i >= total) break;
            root = item_root(W.offset, R.n, i);
            BZ_CHECK(root >= 0 && root < R.n && W.offset[root] <= i && i < W.offset[root + 1], 62);  // item -> root
            uint64_t key;
            depth = root_depth(R, root, key);
            uint64_t me = R.me[root], opp = R.opp[root];
            slot = i - W.offset[root];
            BZ_CHECK(slot < (unsigned)kSlots, 63);  // value slot
            k = 0;
            nodes = 1;
            s_alpha[0] = -kWindow;
            s_beta[0] = kWindow;
            apply_legal(me, opp, kth_bit(legal_mask(me, opp, cells), (int)slot));
            enter(me, opp);
        } else if (!leaf) {  // descend into the next move of level k, row-major
            const uint64_t rem = s_rem[k];
            const uint64_t x = rem & (0ull - rem);
            s_rem[k] = rem ^ x;
            uint64_t me = s_me[k], opp = s_opp[k];
            apply_legal(me, opp, (unsigned)(__ffsll((long long)x) - 1));
            BZ_CHECK(k + 1 < kLevels, 64);  // stack level
            s_alpha[k + 1] = s_alpha[k];
            s_beta[k + 1] = s_beta[k];
            ++k;
            ++nodes;
            enter(me, opp);
        }
        if (!leaf) continue;
        // return v to the parents until one has a move left to search
        while (true) {
            if (k == 0) {
                BZ_CHECK(root * kSlots + slot < R.n * kSlots, 65);  // value slot
                W.vals[root * kSlots + slot] = (int8_t)v;
                atomicAdd(&W.nodes[root], (unsigned long long)nodes);
                k = -1;
                break;
            }
            --k;
            const bool maxing = ((kD0 + k) & 1) == 0;
            int best = s_best[k];
            if (maxing) {
                if (v > best) best = v;
                if (best > s_alpha[k]) s_alpha[k] = best;
            } else {
                if (v < best) best = v;
                if (best < s_beta[k]) s_beta[k] = best;
            }
            s_best[k] = best;
            if (s_alpha[k] >= s_beta[k] || s_rem[k] == 0) {
                v = best;
                continue;
            }
            leaf = false;
            break;
        }
    }
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
    minimax_search_kernel<<<persistent_grid(R.n * 32, kSearchThreads, 8), kSearchThreads, 0, stream>>>(R, cells, W);
    minimax_finish_kernel<<<blocks, 256, 0, stream>>>(R, seed, cells, W, action, value, nodes, nodes_total);
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
