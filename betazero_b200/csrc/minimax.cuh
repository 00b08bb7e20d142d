// Host-side interface of the minimax kernels (minimax.cu) for the other .cu files of the library: bz_minimax_moves reads
// its roots from arrays, the tournament entry (selfplay.cu) from the layout of a tournament ply.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/betazero_b200.h"

namespace bz {

constexpr uint8_t kMinimaxNotSearched = 0xFF;  // entrant_depth of a net entrant

struct MinimaxRoots {
    const uint64_t *me, *opp;  // [n]
    int64_t n;
    // array form (bz_minimax_moves): depth and game key per root
    const uint8_t *depth;
    const uint64_t *key;
    // tournament form (depth == nullptr): root t is searched iff game_of_tree[t] >= 0 and its CTA pair's entrant has a
    // depth; key = key_base + game_of_tree[t]
    const int32_t *game_of_tree;
    const uint8_t *pair_entrant;
    int64_t key_base;
    uint8_t entrant_depth[BZ_MAX_ENTRANTS];  // kMinimaxNotSearched: a net entrant
};

int64_t minimax_workspace_bytes(int64_t n);

// value and nodes (per root) and nodes_total (one int64, added to) may be null
int minimax_launch(const MinimaxRoots &roots, uint64_t seed, int size, void *workspace, uint8_t *action, int8_t *value,
                   int64_t *nodes, int64_t *nodes_total, cudaStream_t stream);

}  // namespace bz
