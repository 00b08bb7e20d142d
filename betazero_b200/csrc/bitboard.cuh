// Bitboard rules for Reversi and tic-tac-toe, device side (sm_100a).
//
// Replaces the reference's grid + ray walk (src/reversi/game_logic/reversi_board.py:25-59,
// src/tic_tac_toe/tic_tac_toe_board.py:20-43) with branch-free 64-bit shift fills.
// bit = row*8 + col.  All functions are pure; one thread handles one board.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bz {

constexpr uint64_t kNotEdgeCols = 0x7E7E7E7E7E7E7E7EULL;  // columns 1..6: horizontal/diagonal fills must not wrap rows

// cells of a size x size board embedded in the 8x8 bit grid
__host__ __device__ constexpr uint64_t cell_mask(int size) {
    return size >= 8 ? ~0ULL : (size == 6 ? 0x00003F3F3F3F3F3FULL : (size == 4 ? 0x000000000F0F0F0FULL : 0ULL));
}

// start position, mover = +1 (X): X on the main diagonal of the centre 2x2 (reversi_board.py:9-11)
__host__ __device__ constexpr uint64_t start_me(int size) {
    return (1ULL << ((size / 2 - 1) * 9)) | (1ULL << ((size / 2) * 9));
}
__host__ __device__ constexpr uint64_t start_opp(int size) {
    return (1ULL << ((size / 2 - 1) * 8 + size / 2)) | (1ULL << ((size / 2) * 8 + size / 2 - 1));
}

// Kogge-Stone fill of `gen` through `pro` in both senses of one axis (shift DIR), returning the
// cells just past each filled run.  Runs are at most 6 long: 1 + 1 + 2 + 2 steps cover them.
template <int DIR>
__device__ __forceinline__ uint64_t axis_moves(uint64_t gen, uint64_t pro) {
    uint64_t up = pro & (gen << DIR), dn = pro & (gen >> DIR);
    up |= pro & (up << DIR);
    dn |= pro & (dn >> DIR);
    const uint64_t pu = pro & (pro << DIR), pd = pro & (pro >> DIR);
    up |= pu & (up << (2 * DIR));
    dn |= pd & (dn >> (2 * DIR));
    up |= pu & (up << (2 * DIR));
    dn |= pd & (dn >> (2 * DIR));
    return (up << DIR) | (dn >> DIR);
}

// K1: all cells where ReversiBoard.is_valid_move(r, c, mover) holds (reversi_board.py:25-41).
__device__ __forceinline__ uint64_t legal_mask(uint64_t me, uint64_t opp, uint64_t cells) {
    const uint64_t inner = opp & kNotEdgeCols;
    uint64_t m = axis_moves<1>(me, inner);
    m |= axis_moves<8>(me, opp);
    m |= axis_moves<7>(me, inner);
    m |= axis_moves<9>(me, inner);
    return m & ~(me | opp) & cells;
}

// discs flipped along one axis by a move on the single-bit board `x`
template <int DIR>
__device__ __forceinline__ uint64_t axis_flips(uint64_t x, uint64_t me, uint64_t pro) {
    uint64_t up = pro & (x << DIR), dn = pro & (x >> DIR);
    up |= pro & (up << DIR);
    dn |= pro & (dn >> DIR);
    const uint64_t pu = pro & (pro << DIR), pd = pro & (pro >> DIR);
    up |= pu & (up << (2 * DIR));
    dn |= pd & (dn >> (2 * DIR));
    up |= pu & (up << (2 * DIR));
    dn |= pd & (dn >> (2 * DIR));
    // a run counts only if the cell just past it holds a mover disc (reversi_board.py:56)
    const uint64_t fu = (me & (up << DIR)) ? up : 0ULL;
    const uint64_t fd = (me & (dn >> DIR)) ? dn : 0ULL;
    return fu | fd;
}

// K2 core: discs flipped by placing on bit `x` (reversi_board.py:49-58).  0 <=> no direction
// brackets anything, which with an empty target cell is exactly "not is_valid_move".
__device__ __forceinline__ uint64_t flips_for(uint64_t x, uint64_t me, uint64_t opp) {
    const uint64_t inner = opp & kNotEdgeCols;
    return axis_flips<1>(x, me, inner) | axis_flips<8>(x, me, opp) | axis_flips<7>(x, me, inner) |
           axis_flips<9>(x, me, inner);
}

struct Applied {
    uint64_t me, opp;  // next mover's view
    bool ok;
};

// make_move + pass with the validity rules of bz_reversi_apply (see include/betazero_b200.h)
__device__ __forceinline__ Applied apply_action(uint64_t me, uint64_t opp, unsigned action, uint64_t cells) {
    Applied r;
    if (action < 64u) {
        const uint64_t x = 1ULL << action;
        const uint64_t f = flips_for(x, me, opp);
        r.ok = (x & ~(me | opp) & cells) != 0 && f != 0;
        r.me = opp & ~f;
        r.opp = me | x | f;
    } else {
        r.ok = action == 64u && legal_mask(me, opp, cells) == 0;
        r.me = opp;
        r.opp = me;
    }
    if (!r.ok) {
        r.me = me;
        r.opp = opp;
    }
    return r;
}

// apply an action already known to be legal (tree descent): no validity work
__device__ __forceinline__ void apply_legal(uint64_t &me, uint64_t &opp, unsigned action) {
    if (action < 64u) {
        const uint64_t x = 1ULL << action;
        const uint64_t f = flips_for(x, me, opp);
        const uint64_t nm = opp & ~f;
        opp = me | x | f;
        me = nm;
    } else {
        const uint64_t t = me;
        me = opp;
        opp = t;
    }
}

// the cell of the k-th set bit of m in ascending cell order (k < popcount(m))
__device__ __forceinline__ unsigned kth_bit(uint64_t m, int k) {
    for (; k > 0; --k) m &= m - 1;
    return (unsigned)(__ffsll((long long)m) - 1);
}

// a move drawn from the legal moves m (m != 0) by the 32-bit draw u: the k-th legal move in ascending cell order,
// k = floor(u * moves / 2^32)
__device__ __forceinline__ unsigned pick_move(uint64_t m, uint32_t u) {
    return kth_bit(m, (int)(((uint64_t)u * (uint64_t)__popcll(m)) >> 32));
}

// ---- group-cooperative forms (tree kernels: a group of G lanes owns one board) -------------------
// The 8 ray directions are spread over 8 lanes of the group instead of being computed serially by
// every lane: group lane d handles shift {1,7,8,9}[d & 3]; lanes 4..7 work on the bit-reversed
// board, where the ">>" senses become "<<", so all lanes run the same left-shift code with a
// per-lane shift count.  Results are combined with redux.sync OR over the group's lanes.
// G in {8, 16, 32}; gmask = the group's lanes, gl = lane index inside the group.
// A whole warp: redux.sync.  Sub-warp groups: a redux with a different member mask per group is serialised group
// by group (ncu: 12 % of the wave kernel's stall samples), so the groups use an xor butterfly over the full warp
// instead (lane ^ d stays inside an aligned group of 8 or 16 lanes).  Every lane of the warp must call this together.
// G: the group size as a compile-time constant (the butterfly is then straight-line code; as a loop over a run-time
// popc(gmask) it was three trips with a branch each, on the critical path of every leaf)
template <int G>
__device__ __forceinline__ uint64_t group_or64(unsigned gmask, uint64_t v) {
    unsigned lo = (unsigned)v, hi = (unsigned)(v >> 32);
    if (G == 32) {
        lo = __reduce_or_sync(0xFFFFFFFFu, lo);
        hi = __reduce_or_sync(0xFFFFFFFFu, hi);
    } else {
#pragma unroll
        for (int d = G >> 1; d; d >>= 1) {
            lo |= __shfl_xor_sync(0xFFFFFFFFu, lo, d);
            hi |= __shfl_xor_sync(0xFFFFFFFFu, hi, d);
        }
    }
    (void)gmask;
    return ((uint64_t)hi << 32) | lo;
}

// one-directional Kogge-Stone fill of gen through pro with left shift s (runs <= 6)
__device__ __forceinline__ uint64_t fill_left(uint64_t gen, uint64_t pro, int s) {
    uint64_t f = pro & (gen << s);
    f |= pro & (f << s);
    const uint64_t pp = pro & (pro << s);
    f |= pp & (f << (2 * s));
    f |= pp & (f << (2 * s));
    return f;
}

__device__ __forceinline__ int lane_shift(int gl) {
    const int k = gl & 3;  // 1, 7, 8, 9
    return k == 0 ? 1 : 6 + k;
}

// discs flipped by the move on single-bit board x; every lane of the group returns the full set
template <int G>
__device__ __forceinline__ uint64_t group_flips(unsigned gmask, int gl, uint64_t x, uint64_t me, uint64_t opp) {
    const int s = lane_shift(gl);
    const bool rev = gl & 4;
    uint64_t g = x, m = me, o = opp;
    if (rev) { g = __brevll(g); m = __brevll(m); o = __brevll(o); }
    const uint64_t pro = (s == 8) ? o : (o & kNotEdgeCols);
    uint64_t f = fill_left(g, pro, s);
    f = (m & (f << s)) ? f : 0ULL;  // the run must end on a mover disc (reversi_board.py:56)
    if (rev) f = __brevll(f);
    if (gl >= 8) f = 0ULL;
    return group_or64<G>(gmask, f);
}

// candidate moves (before the empty-cell mask) of `gen` against `pro` in direction lane gl & 7
__device__ __forceinline__ uint64_t dir_moves(int gl, uint64_t gen, uint64_t o) {
    const int s = lane_shift(gl);
    const bool rev = gl & 4;
    if (rev) { gen = __brevll(gen); o = __brevll(o); }
    const uint64_t pro = (s == 8) ? o : (o & kNotEdgeCols);
    uint64_t mv = fill_left(gen, pro, s) << s;
    if (rev) mv = __brevll(mv);
    return mv;
}

// legal cells of the mover (me) and of the opponent; every lane of the group returns both masks.
// G >= 16: lanes 0..7 mover, 8..15 opponent, one pass.  G == 8: two passes over the same 8 lanes.
template <int G>
__device__ __forceinline__ void group_legal_masks(unsigned gmask, int gl, uint64_t me, uint64_t opp, uint64_t cells,
                                                  uint64_t &mask_me, uint64_t &mask_opp) {
    const uint64_t empty = ~(me | opp) & cells;
    if (G >= 16) {
        const bool second = gl & 8;
        const uint64_t mv = dir_moves(gl, second ? opp : me, second ? me : opp);
        mask_me = group_or64<G>(gmask, (gl < 8) ? mv : 0ULL) & empty;
        mask_opp = group_or64<G>(gmask, (gl >= 8 && gl < 16) ? mv : 0ULL) & empty;
    } else {
        mask_me = group_or64<G>(gmask, dir_moves(gl, me, opp)) & empty;
        mask_opp = group_or64<G>(gmask, dir_moves(gl, opp, me)) & empty;
    }
}

// The same for G == 8 with the opponent's mask computed only when some group of the warp needs it: the caller uses
// mask_opp only where mask_me == 0 (pass or game over?), which few positions are, and `want` is false for groups whose
// result is discarded.  Every lane of the warp must call this together; mask_opp is valid where want && mask_me == 0.
__device__ __forceinline__ void group8_legal_masks_lazy(unsigned gmask, int gl, uint64_t me, uint64_t opp, uint64_t cells,
                                                        bool want, uint64_t &mask_me, uint64_t &mask_opp) {
    const uint64_t empty = ~(me | opp) & cells;
    mask_me = group_or64<8>(gmask, dir_moves(gl, me, opp)) & empty;
    mask_opp = 0;
    if (__any_sync(0xFFFFFFFFu, want && mask_me == 0)) mask_opp = group_or64<8>(gmask, dir_moves(gl, opp, me)) & empty;
}

// ---- tic-tac-toe: 9-bit boards, bit = row*3 + col --------------------------------------------
__device__ __forceinline__ bool ttt_has_line(unsigned b) {
    // rows 0x007 0x038 0x1C0, columns 0x049 0x092 0x124, diagonals 0x111 0x054
    return ((b & 0x007u) == 0x007u) | ((b & 0x038u) == 0x038u) | ((b & 0x1C0u) == 0x1C0u) |
           ((b & 0x049u) == 0x049u) | ((b & 0x092u) == 0x092u) | ((b & 0x124u) == 0x124u) |
           ((b & 0x111u) == 0x111u) | ((b & 0x054u) == 0x054u);
}

}  // namespace bz
