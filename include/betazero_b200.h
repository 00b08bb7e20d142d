/*
 * betazero_b200.h -- C ABI of the B200-native self-play engine for whaiproject/BetaZero.
 *
 * The reference is pure Python with no FFI layer; its drop-in boundary is the duck-typed board /
 * player API (SURVEY.md section 8b).  This header is the boundary a native binding for that API
 * would use: plain `extern "C"`, pointers + sizes, no torch / Python types.  Each entry point
 * cites the reference code whose computation it replaces (paths relative to the reference root).
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer (sm_100a, B200) unless a parameter says "host".
 *  - Every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default
 *    stream), never allocates, never synchronises, never throws.  The caller owns all buffers.
 *  - Return value: BZ_OK (0), BZ_ERR_ARG for a bad argument, or -(1000 + cudaError_t).
 *  - Reversi boards are SoA uint64 pairs, MOVER-RELATIVE: `me` = discs of the side to move,
 *    `opp` = the other side's.  bit = row*8 + col for every board size (4, 6, 8); cells
 *    outside size x size are never set.  The reference's absolute view (`.board` with +1 = X,
 *    -1 = O, reversi_board.py:7-11) is X = (player == +1 ? me : opp).
 *  - Reversi action ids: a = row*8 + col, 64 = pass.  Policy vectors have BZ_REVERSI_ACTIONS
 *    (65) entries.  Tic-tac-toe: a = row*3 + col, 9 entries.
 *  - There is no CPU fallback anywhere behind this ABI.
 */
#ifndef BETAZERO_B200_H
#define BETAZERO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BZ_OK 0
#define BZ_ERR_ARG (-1)
#define BZ_ERR_UNALIGNED (-2)
#define BZ_ABI_VERSION 6

#define BZ_REVERSI_ACTIONS 65
#define BZ_TTT_ACTIONS 9
#define BZ_PASS 64

#define BZ_GAME_REVERSI 0
#define BZ_GAME_TTT 1

typedef void *bz_stream_t; /* cudaStream_t */

int bz_abi_version(void);

/* Process-wide switch for programmatic dependent launch between bz_mcts_step and bz_mlp_forward_pair*
 * (each kernel's prologue overlaps the other's tail; both wait on griddepcontrol before reading
 * the other's output).  Returns the previous setting.  Off by default. */
int bz_set_pdl(int enable);
/* static string for a return code of this library (host) */
const char *bz_error_string(int code);

/* ------------------------------------------------------------------------------------------
 * Reversi environment (kernels K1..K3 of SURVEY.md section 2.1)
 * ---------------------------------------------------------------------------------------- */

/* Start position for n boards: ReversiBoard.__init__, reversi_board.py:4-11, plus
 * `current_player = 1` of ReversiTerminal.__init__, reversi_terminal.py:14.
 * player may be NULL.  size in {4, 6, 8}. */
int bz_reversi_init(uint64_t *me, uint64_t *opp, int8_t *player, int64_t n, int size, bz_stream_t stream);

/* K1.  mask bit (r*8+c) == ReversiBoard.is_valid_move(r, c, mover) for all cells, i.e.
 * generate_possible_moves(mover): reversi_board.py:25-41, 87-88.  24 B/board. */
int bz_reversi_legal_mask(const uint64_t *me, const uint64_t *opp, uint64_t *mask, int64_t n, int size,
                          bz_stream_t stream);

/* K2.  ReversiBoard.make_move(r, c, mover), reversi_board.py:43-59, with the result expressed
 * for the NEXT mover (me_out = old opp after flips, opp_out = old me + placed + flipped).
 * action 64 = pass: board unchanged, sides swap (reversi_terminal.py:31-35).
 * err[i] = 1 where the reference raises ValueError("Invalid move") (reversi_board.py:44-45), or
 * for a pass while the mover has a move; the board is then copied through UNCHANGED and
 * UNSWAPPED.  err may be NULL.  33 B/board (+1 with err). */
int bz_reversi_apply(const uint64_t *me, const uint64_t *opp, const uint8_t *action, uint64_t *me_out,
                     uint64_t *opp_out, uint8_t *err, int64_t n, int size, bz_stream_t stream);

/* K3.  over = ReversiBoard.is_game_over() (reversi_board.py:61-65); winner_for_me / counts =
 * get_score() (reversi_board.py:67-76) seen from the mover: +1 mover has more discs, -1 fewer,
 * 0 tie.  Reported for every board (get_score does not require a finished game).  Any output
 * pointer may be NULL.  20 B/board. */
int bz_reversi_terminal(const uint64_t *me, const uint64_t *opp, uint8_t *over, int8_t *winner_for_me,
                        uint8_t *cnt_me, uint8_t *cnt_opp, int64_t n, int size, bz_stream_t stream);

/* K1+K2 fused: one ply of the reference episode loop (reversi_terminal.py:22-35) with the
 * deterministic "first legal move" player: mask = legal moves; action = lowest set bit of mask,
 * or 64 (pass) when mask == 0; boards advance to the next mover's view.  mask_out / action_out
 * may be NULL.  41 B/board. */
int bz_reversi_step_first_legal(const uint64_t *me, const uint64_t *opp, uint64_t *mask_out, uint8_t *action_out,
                                uint64_t *me_out, uint64_t *opp_out, int64_t n, int size, bz_stream_t stream);

/* K6 (stand-alone form).  Canonical network input, side to move = +1
 * (players.py:85 `symbol * board`; generate_training_games.py:17-18): bf16 planes
 * [n, 2, 8, 8], plane 0 = me, plane 1 = opp, 1.0 / 0.0.  16 B in + 256 B out per board. */
int bz_reversi_planes(const uint64_t *me, const uint64_t *opp, void *planes_bf16, int64_t n, bz_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Tic-tac-toe environment (K4).  Absolute 9-bit boards x (+1) and o (-1), bit = row*3 + col.
 * ---------------------------------------------------------------------------------------- */

/* TicTacToeBoard.generate_possible_moves(), tic_tac_toe_board.py:42-43 (== is_valid_move :20-21) */
int bz_ttt_legal_mask(const uint16_t *x, const uint16_t *o, uint16_t *mask, int64_t n, bz_stream_t stream);

/* TicTacToeBoard.make_move(r, c, player), tic_tac_toe_board.py:23-29; err = ValueError. */
int bz_ttt_apply(const uint16_t *x, const uint16_t *o, const uint8_t *action, const int8_t *player,
                 uint16_t *x_out, uint16_t *o_out, uint8_t *err, int64_t n, bz_stream_t stream);

/* TicTacToeBoard.is_game_over(), tic_tac_toe_board.py:31-40: lines of +1 are tested before
 * lines of -1, then the full-board draw.  winner = +1 / -1 / 0, or 2 for Python's None. */
int bz_ttt_terminal(const uint16_t *x, const uint16_t *o, uint8_t *over, int8_t *winner, int64_t n,
                    bz_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Batched MCTS (K5..K8).  The reference has no MCTS; the semantics are those frozen in
 * oracle/mcts_ref.py, and the entry point this serves is Player.get_move(board) -> (row, col)
 * (reversi_players.py:5-8, players.py:6-9).
 *
 * One warp owns one tree.  All pools are caller-allocated SoA arrays resident in HBM.
 * Tree-local indices are int32; a tree's slice of a per-edge array starts at
 * (int64)tree * edge_cap.
 * ---------------------------------------------------------------------------------------- */

/* Tree storage.  Each tree owns an ARENA of 32-bit words; an expanded node is one contiguous,
 * 32-byte aligned NODE BLOCK inside it, SoA within the block so that lane i of the owning warp
 * reads edge i of every field with one coalesced access and a whole node costs one short burst
 * of adjacent DRAM sectors:
 *
 *     word 0..1  me      (uint64, board of the node for its mover)
 *     word 2..3  opp
 *     word 4     n       (number of edges, 1..33)
 *     word 5..7  reserved
 *     word 8      .. 8+n-1    N[n]     int32   visit counts
 *     word 8+n    .. 8+2n-1   W[n]     float32 total value
 *     word 8+2n   .. 8+3n-1   P[n]     float32 prior
 *     word 8+3n   .. 8+4n-1   meta[n]  uint32  action + child reference
 *     (padded to a multiple of 8 words)
 *
 * meta: bits 0..6 action, bits 7..12 number of edges of the child (0 = child is not a normal
 * node), bits 13..31 the child's block offset in 8-word units.  With child_n == 0 the offset
 * field holds BZ_META_UNEXPANDED, or BZ_META_TERMINAL + {0,1,2} for a terminal child worth
 * {-1, 0, +1} to ITS side to move.  Because an edge carries its child's (offset, n), one level of
 * the PUCT descent is a single round of dependent loads. */
#define BZ_NODE_HEADER_WORDS 8
#define BZ_META_OFF_SHIFT 13
#define BZ_META_N_SHIFT 7
#define BZ_META_UNEXPANDED 0x7FFFFu
#define BZ_META_TERMINAL 0x7FFF0u
#define BZ_MAX_ARENA_UNITS 0x7FFF0 /* 8-word units per tree (16.7 MB) */
#define BZ_MAX_NODE_UNITS 18       /* worst case: 33 edges -> 8 + 132 words -> 18 units */

#define BZ_MAX_LEAVES 8 /* pools.n_leaves */

/* leaf_status values */
#define BZ_LEAF_EVAL 0     /* needs the evaluator's output */
#define BZ_LEAF_TERMINAL 1 /* game over at the leaf: value known, evaluator output ignored */
#define BZ_LEAF_ERROR 2    /* pool overflow / no pending leaf; iteration skipped */

/* how bz_mcts_expand_backup / bz_mcts_step read the evaluator's output */
#define BZ_PRIOR_WEIGHTS 0 /* eval_out: float32 [n_trees, n_actions] weights >= 0, value: float32 [n_trees].
                              P = w / sum over legal (ascending action order; sum 0 -> uniform).
                              The parity mode: bit-exact against the oracle. */
#define BZ_PRIOR_LOGITS_BF16 1 /* eval_out: bf16 [n_trees, eval_stride] raw network output: columns
                              0..n_actions-1 policy logits, column n_actions the pre-tanh value.
                              The kernel computes the softmax over the LEGAL actions and tanh itself
                              (fast path: no softmax / cast / copy launches); `value` is ignored. */

typedef struct bz_tree_pools {
    int32_t game;        /* BZ_GAME_REVERSI / BZ_GAME_TTT */
    int32_t board_size;  /* Reversi: 4, 6, 8 */
    int32_t n_trees;
    int32_t n_actions;   /* 65 / 9: row length of weight / count / pi rows */
    int32_t arena_units; /* 8-word units per tree (<= BZ_MAX_ARENA_UNITS); 18 per iteration never overflows */
    int32_t max_depth;   /* path capacity per tree */
    float c_puct;
    int32_t prior_mode;  /* BZ_PRIOR_WEIGHTS / BZ_PRIOR_LOGITS_BF16 */
    int32_t eval_stride; /* row stride (elements) of eval_out in logits mode (>= n_actions + 1) */
    int32_t group_lanes; /* lanes that own one tree: 32 (warp per tree), 16, 8 (4 trees per warp), 0 = choose by n_trees */
    int32_t n_leaves;    /* 0 / 1: one leaf per tree and iteration (the bit-exact parity definition).  K in 2..BZ_MAX_LEAVES:
                            K descents per tree and iteration with VIRTUAL LOSS (a descent leaves N += 1, W -= 1 on its
                            edges until its backup): the pending-leaf arrays below then hold K * n_trees entries, slot-major
                            (entry slot * n_trees + tree), eval_out / value have K * n_trees rows, and an iteration counts
                            K simulations.  K = 2 / 4 with group_lanes 0 or 32 run in "wave mode" (the K descents are the
                            32/K-lane groups of the tree's warp, one level apart); other combinations handle the slots one
                            after the other.  Definition and oracle: oracle/mcts_ref.py MCTS.select_vl / expand_backup_vl. */
    /* per tree [n_trees] */
    uint64_t *root_me, *root_opp;
    uint32_t *root_meta;  /* like an edge's meta, for the (virtual) edge into the root */
    int32_t *arena_used;  /* bump allocator, in units */
    int32_t *edge_count;  /* edges created since reset (mean children b of the roofline model) */
    int32_t *sim_count;   /* completed select/expand iterations since reset */
    int32_t *depth_sum;   /* sum of path lengths of those iterations (mean depth d) */
    int32_t *error;       /* sticky: 1 = arena overflow, 2 = path overflow */
    /* the arenas: uint32 [n_trees * arena_units * 8] */
    uint32_t *arena;
    /* pending leaf, per tree */
    uint32_t *path;        /* [rows * max_depth * 4] records {word index of N, n, N, W bits}, root first; rows = n_trees * max(n_leaves, 1) */
    int32_t *path_len;     /* [rows] (and so on for every leaf_* array) */
    int32_t *leaf_parent;  /* arena word index of the meta of the edge into the leaf (-1: the leaf is the root) */
    uint64_t *leaf_me, *leaf_opp;
    uint64_t *leaf_mask;   /* legal cells of the leaf's mover (0 with status EVAL = the mover must pass) */
    uint8_t *leaf_status;
    uint8_t *leaf_action;  /* action of the edge into the leaf */
    float *leaf_value;     /* terminal value for the leaf's mover */
    void *leaf_planes;     /* bf16 [rows, 2, 8, 8] canonical planes of the leaf (K6); TTT: [rows, 9] */
} bz_tree_pools;

/* Empty every tree and set its root position (mover-relative). */
int bz_mcts_reset(const bz_tree_pools *pools, const uint64_t *root_me, const uint64_t *root_opp,
                  bz_stream_t stream);

/* K5 (+K6 fused): one PUCT descent per tree.  Writes path/path_len, the leaf board, its status
 * and its canonical bf16 planes. */
int bz_mcts_select(const bz_tree_pools *pools, bz_stream_t stream);

/* K6 on its own: re-pack leaf_me/leaf_opp into leaf_planes (select already does this). */
int bz_mcts_gather(const bz_tree_pools *pools, bz_stream_t stream);

/* K7: expand the pending leaf with the evaluator's output (see prior_mode) and back the leaf
 * value (for the leaf's mover) up the path: store-only, atomic-free, one lane per path edge.
 * Terminal leaves back up their exact game result instead. */
int bz_mcts_expand_backup(const bz_tree_pools *pools, const void *eval_out, const float *value,
                          bz_stream_t stream);

/* K7+K5+K6 in one launch: finish iteration i with the evaluator's output, start iteration i+1. */
int bz_mcts_step(const bz_tree_pools *pools, const void *eval_out, const float *value, bz_stream_t stream);

/* The whole search of one move in ONE launch: K5 (select), then n_iterations x [the policy/value MLP on the pending
 * leaves, K7 (expand + backup), K5 + K6 for the next iteration (not after the last)] -- the sequence
 * bz_mcts_select, n x [bz_mlp_forward_pair*, bz_mcts_step / bz_mcts_expand_backup] computes, with bit-identical trees.
 * Player.get_move's search loop (reversi_players.py:5-8) without a kernel boundary per iteration: a CTA pair owns 56
 * trees in two islands; while one island's leaves are in the net (tcgen05 cta_group::2, the weight image of
 * bz_mlp_forward_pair resident in shared memory for the whole search, the leaf planes written from registers into the
 * A operand) the other island's warps walk their trees.
 * Shape: Reversi; n_leaves == 2 or 4 in wave mode (group_lanes 0 or 32) or n_leaves <= 1 (the sequential one-leaf search: a
 * warp per tree here whatever group_lanes says -- the trees do not depend on it); prior_mode BZ_PRIOR_LOGITS_BF16 with
 * eval_stride == 72 (BZ_ERR_ARG otherwise: use the per-iteration entry points).  One launch holds 148 * 28 = 4144
 * trees; more trees are searched in equal chunks, one launch after the other on the stream.
 * eval_out: ignored (may be NULL; earlier versions used it as scratch -- the net's rows now stay in shared memory);
 * leaf_planes is not written.  n_iterations = simulations per tree / max(n_leaves, 1). */
int bz_mcts_search_fused(const bz_tree_pools *pools, const void *weight_image_pair, void *eval_out, int n_iterations,
                         bz_stream_t stream);

/* bz_mcts_search_fused with an entrant table (tournaments: many nets and search budgets in one launch): the 56 trees
 * [56 p, 56 p + 56) of the pools are searched with images[e] for n_iterations[e] iterations, e = pair_entrant[p].
 * images / n_iterations: host arrays of n_entrants (1 .. BZ_MAX_ENTRANTS) entries, copied into the launch; an image may
 * appear under several entrants.  pair_entrant: device uint8 [ceil(n_trees / 56)], counted from tree 0 of the pools
 * whatever the chunking (e.g. written by bz_tournament_layout); an entry >= n_entrants is a bounds-check failure
 * (BZ_CHECK) and its trees are left as they are, as are the trees of an entrant with 0 iterations.  A pair's trees are
 * bit-identical to a bz_mcts_search_fused of the same roots with images[e] and n_iterations[e].  The pools' arena must
 * hold the largest budget.  A launch lasts as long as its largest count: pairs with fewer iterations leave their SMs idle
 * once they are done.  BZ_ERR_ARG: n_entrants out of range, a NULL image, a negative count, pair_entrant == NULL;
 * BZ_ERR_UNALIGNED: an image not 16-byte aligned. */
#define BZ_MAX_ENTRANTS 64
int bz_mcts_search_fused_entrants(const bz_tree_pools *pools, const void *const *images, const int32_t *n_iterations,
                                  int n_entrants, const uint8_t *pair_entrant, bz_stream_t stream);

/* Tree reuse across moves (opt-in; the default -- bz_mcts_reset before every search -- is what the goldens pin).
 * After the game of tree t has played action[t] and stands at (new_me[t], new_opp[t]), mover-relative for the side to
 * move there, the tree is re-rooted at the child that action leads to: the child's subtree -- statistics, priors,
 * shape -- is compacted to the front of the tree's arena and becomes the tree; sim_count[t] becomes the visit count of
 * the edge into the new root.  The subtree is kept iff the root has an edge for action[t], the child behind it has
 * been expanded, the child's board equals the new position (a slot whose game ended and restarted therefore starts an
 * empty tree) and the subtree occupies at most cap_units arena units; otherwise the tree is emptied at the new
 * position exactly as bz_mcts_reset would (cap_units * 8 + cap_units / 2 + 1 <= arena_units * 8, BZ_ERR_ARG otherwise:
 * the top of the scratch arena is the copy's queue).  Choose cap_units <= arena_units - 18 * (simulations of the next search):
 * then the next search cannot overflow the arena.  The next search (bz_mcts_search_fused, or select / step ...) adds its
 * simulations to the kept statistics, as AlphaZero's self-play does; Player.get_move (reversi_players.py:5-8) sees
 * visit counts that include the inherited ones.
 * scratch_arena: uint32 [n_trees * arena_units * 8], 32-byte aligned (contents are scratch).  inherited (may be NULL):
 * int32 [n_trees], the visits each new root starts with (0: empty tree).  Definition: oracle/mcts_ref.py MCTS.advance. */
int bz_mcts_reroot(const bz_tree_pools *pools, void *scratch_arena, const uint8_t *action, const uint64_t *new_me,
                   const uint64_t *new_opp, int cap_units, int32_t *inherited, bz_stream_t stream);

/* Root exploration noise (AlphaZero self-play; OFF in every parity test): for each tree whose
 * root is expanded, P[e] <- (1 - eps) * P[e] + eps * noise[a_e] / sum over the root's edges of
 * noise[a].  noise: float32 [n_trees, n_actions] > 0 (e.g. Gamma(alpha, 1) samples: the
 * normalised vector is then Dirichlet(alpha) over the legal moves).  Call after the iteration that
 * expanded the root and before the next select. */
int bz_mcts_root_noise(const bz_tree_pools *pools, const float *noise, float eps, bz_stream_t stream);

/* Read one tree's root edges back in action order (debug / tests): N, W, P scattered by action
 * into rows of n_actions (zeros elsewhere).  Any output may be NULL. */
int bz_mcts_root_edges(const bz_tree_pools *pools, int32_t *N, float *W, float *P, bz_stream_t stream);

/* K8: root visit counts (int32 [n_trees, n_actions]), pi = N / sum N and q = W / N (float32,
 * same shape; either may be NULL), scattered by action, zeros elsewhere. */
int bz_mcts_root_policy(const bz_tree_pools *pools, int32_t *visit_counts, float *pi, float *q,
                        bz_stream_t stream);

/* Most-visited action per tree, lowest action id on ties (the argmax-over-legal pick of
 * players.py:92-98 applied to visit counts); 255 if the root has no visits. */
int bz_mcts_best_action(const bz_tree_pools *pools, uint8_t *action, bz_stream_t stream);

/* Parity-mode evaluator: deterministic integer-hash "pseudo-net" on (me, opp); weights 1..32
 * and value k/8 are exact in fp32, identical to oracle/mcts_ref.py:hash_eval. */
int bz_hash_eval(const uint64_t *me, const uint64_t *opp, uint64_t salt, int n_actions, float *prior_w,
                 float *value, int64_t n, bz_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Lockstep self-play driver state (the batched form of the reference episode loops,
 * reversi_terminal.py:16-38: search -> move or pass -> terminal test -> flip player; finished
 * games are scored with get_score (reversi_board.py:67-76), flushed to the replay buffer and
 * their slot restarts from the start position with a fresh game id).
 * ---------------------------------------------------------------------------------------- */
typedef struct bz_selfplay_state {
    int32_t n_games;    /* slots == trees of the pools used with it */
    int32_t board_size; /* 4, 6, 8 */
    int32_t max_plies;  /* history rows per slot (>= 2*cells; 128 for 8x8) */
    int32_t temp_plies; /* plies < temp_plies sample the move ~ visit counts (Philox keyed by
                           seed, game id, ply); later plies take the most visited action */
    uint64_t seed;
    int64_t id_stride;  /* a restarted slot continues with game_id + id_stride */
    int64_t replay_cap; /* records */
    /* per slot [n_games] */
    uint64_t *me, *opp; /* current position, mover-relative */
    int8_t *player;     /* absolute side to move: +1 = X, -1 = O */
    int32_t *ply;
    int64_t *game_id;
    /* per slot history [n_games * max_plies] (pi: [.., 65]) */
    uint64_t *hist_me, *hist_opp;
    int8_t *hist_player;
    uint8_t *hist_action;
    float *hist_pi;
    /* replay buffer [replay_cap] (pi: [replay_cap, 65]); z = game result for the record's mover */
    uint64_t *rp_me, *rp_opp;
    float *rp_pi;
    int8_t *rp_z;
    int64_t *rp_game;
    int16_t *rp_ply;
    /* device counters, uint64 [8]: 0 replay records COMMITTED (rows [0, counters[0]) of rp_* are all valid: a
     * finished game reserves its rows atomically and takes none if it does not fit), 1 plies played, 2 O wins,
     * 3 draws, 4 X wins, 5 records dropped (replay full), 6 games finished, 7 reserved */
    unsigned long long *counters;
} bz_selfplay_state;

/* All slots to the start position (ReversiBoard.__init__, reversi_board.py:9-11; X moves first,
 * reversi_terminal.py:14); slot s gets game id first_game_id + s.  Zeroes the counters. */
int bz_selfplay_init(const bz_selfplay_state *st, int64_t first_game_id, bz_stream_t stream);

/* One lockstep ply for every slot, from the finished search in `pools` (tree s <-> slot s):
 * pi = root visit counts / total, action = sampled or most visited (lowest id on ties), record
 * to history, apply (K2), terminal test (K3); a finished game is flushed to the replay buffer
 * with z and the slot restarts.  action_out (uint8 [n_games]) may be NULL. */
int bz_selfplay_advance(const bz_selfplay_state *st, const bz_tree_pools *pools, uint8_t *action_out,
                        bz_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Batched round-robin tournaments: every pairing of up to BZ_MAX_ENTRANTS entrants (a net and a search budget each) in
 * the same launches; a net-versus-net match is the tournament of two entrants and the one pairing (0, 1).  Game pair i
 * is pairing (first[i], second[i]): both games play the same random opening (pair id first_pair_id + i), then `first`
 * is X in game 2i and O in game 2i+1.  Every ply: bz_tournament_layout puts each entrant's movers into contiguous,
 * pair-aligned tree ranges, bz_mcts_reset + bz_mcts_search_fused_entrants search them, bz_match_advance plays the most
 * visited root action (lowest action on ties) in every live game and scores finished games (get_score,
 * reversi_board.py:67-76).  bz_match_init and bz_match_advance take the tournament state's `match`.
 * ---------------------------------------------------------------------------------------- */
#define BZ_MATCH_RUNNING 2       /* result of a game that has not ended */
#define BZ_MATCH_MAX_PLIES 128   /* rows of `moves` per game */
#define BZ_MATCH_TREES_PER_PAIR 56
typedef struct bz_match_state {
    int32_t n_games;       /* even, < 65536 */
    int32_t board_size;    /* 4, 6, 8 */
    int32_t opening_plies; /* uniformly random legal moves (Philox keyed by seed, pair id, ply) before the nets play */
    int32_t n_trees;       /* rows of the tree-ordered arrays: >= n_games + 55 */
    uint64_t seed;
    int64_t first_pair_id; /* pair i draws its opening with pair id first_pair_id + i */
    /* per game [n_games] */
    uint64_t *me, *opp;    /* current position, mover-relative */
    int8_t *player;        /* absolute side to move: +1 = X, -1 = O */
    int32_t *ply;
    int8_t *result;        /* BZ_MATCH_RUNNING, or the winner: +1 X, -1 O, 0 draw */
    uint8_t *count_x, *count_o; /* final disc counts (0 while running) */
    uint8_t *moves;        /* [n_games * BZ_MATCH_MAX_PLIES], action of each ply (64 = pass), 255 after the end */
    int32_t *tree_of_game; /* tree searched for the game this ply, -1 once it has ended */
    /* per tree [n_trees] (the layout of the current ply) */
    int32_t *game_of_tree; /* -1: padding, or past the trees searched this ply */
    uint64_t *root_me, *root_opp; /* the bz_mcts_reset roots (padding: an empty board, a finished game) */
    uint8_t *pair_net;     /* [ceil(n_trees / 56)]: entrant ids, the pair_entrant of bz_mcts_search_fused_entrants */
    /* int64 [8]: 0 live games, 1 trees to search this ply, 2 padding trees this ply (0..2 written by
     * bz_tournament_layout), 3 finished games, 4 wins, 5 draws, 6 losses and 7 disc difference, all four summed over
     * every pairing from its `first` entrant's point of view */
    int64_t *counters;
} bz_match_state;

/* Every game to the start position, then the opening; games that end inside it are scored.  Zeroes the counters. */
int bz_match_init(const bz_match_state *st, bz_stream_t stream);
/* One ply of every live game from the finished search in `pools` (n_trees == st->n_trees; the trees bz_tournament_layout
 * assigned): most visited root action, lowest action id on ties (the first legal move, or a pass, if the root has no
 * visits); record, apply, terminal test, score. */
int bz_match_advance(const bz_match_state *st, const bz_tree_pools *pools, bz_stream_t stream);

typedef struct bz_tournament_state {
    bz_match_state match;  /* games, openings, moves, results, the layout of the current ply */
    int32_t n_entrants;    /* 1 .. BZ_MAX_ENTRANTS */
    uint8_t *first, *second; /* per game pair [n_games / 2]: `first` is X in game 2i and O in game 2i+1 */
} bz_tournament_state;

/* The tree layout of this ply (one CTA): a stable partition of the live games by the entrant to move -- entrants in id
 * order, games in game order inside an entrant, every non-empty range but the last padded with empty boards to the next
 * multiple of 56.  Writes tree_of_game, game_of_tree, root_me / root_opp, pair_net (entrant ids; pairs past the searched
 * prefix: the last entrant with movers) and counters 0..2.  BZ_ERR_ARG: a bad match state, n_entrants out of range, NULL
 * first / second, match.n_trees < n_games + 55 (n_entrants - 1).  An entrant id >= n_entrants in first / second is a
 * bounds-check failure (BZ_CHECK); such a game gets no tree. */
int bz_tournament_layout(const bz_tournament_state *st, bz_stream_t stream);

/* Minimax entrants (the reference's depth-limited OptimalPlayer, reversi_players.py:35-77, and RandomPlayer as its depth 0;
 * see bz_minimax_moves).  entrant_depth: a host array of n_entrants entries, -1 for a net entrant, 0 .. BZ_MINIMAX_MAX_DEPTH
 * for a minimax entrant.  A minimax entrant keeps its range of trees in bz_tournament_layout and is given 0 iterations in
 * bz_mcts_search_fused_entrants (its trees are then not touched).
 * bz_tournament_minimax: for every tree t < match.n_trees of a minimax entrant's range that holds a game g
 * (game_of_tree[t] >= 0), action[t] = the bz_minimax_moves move of the root (root_me[t], root_opp[t]) at the entrant's
 * depth with the match's seed and key 2 first_pair_id + g; action[t] = 255 for every other tree.  workspace:
 * bz_minimax_workspace_bytes(match.n_trees) bytes, 16-byte aligned.  nodes_total (may be NULL): device int64 [1], the
 * nodes searched are added to it.
 * bz_tournament_advance: bz_match_advance for tournaments with minimax entrants -- the game of a minimax entrant's tree
 * plays action[t], every other game exactly what bz_match_advance plays.  pools may be NULL when every entrant is minimax.
 * BZ_ERR_ARG (both): a bad tournament state, an entry of entrant_depth out of range, a NULL action or workspace; and for
 * bz_tournament_advance a NULL or mismatched pools with a net entrant. */
int bz_tournament_minimax(const bz_tournament_state *st, const int32_t *entrant_depth, void *workspace, uint8_t *action,
                          int64_t *nodes_total, bz_stream_t stream);
int bz_tournament_advance(const bz_tournament_state *st, const bz_tree_pools *pools, const int32_t *entrant_depth,
                          const uint8_t *action, bz_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Depth-limited minimax: the reference's OptimalPlayer.get_move (src/reversi/players/reversi_players.py:35-77; the
 * definition is oracle/minimax_ref.py).  For every root i (mover-relative (me[i], opp[i]), the mover is the player):
 *  - minimax(node, depth): if depth >= max_depth or the game is over (reversi_board.py:61-65), the disc difference from
 *    the player's point of view (evaluate_board via get_score, :71-77; no win bonus).  Otherwise the player's nodes
 *    (even depths) take the maximum over their moves in row-major order, the opponent's nodes the minimum (:50-69).
 *  - No pass handling: a node whose side has no move in a game that is not over is worth -inf at the player's nodes and
 *    +inf at the opponent's (the loops of :51-59 and :61-69 never run).  value = +-127 stands for +-inf.
 *  - The move is the first root move whose value is strictly above every earlier one (:56-58).  When there is none --
 *    depth[i] == 0, or every child is worth -inf -- the move is drawn as the reference's random.choice (:42-43) is, here
 *    reproducibly: u = Philox4x32-10(seed, key 2^32 + key[i], counter popcount(me | opp)), the k-th legal move in
 *    ascending cell order with k = floor(u * moves / 2^32).  RandomPlayer (:26-32) is depth 0.
 *  - action: the move (row*8 + col), 64 when the player has no move (a pass), 255 when the game is over.  value: the
 *    root's minimax value (int8).  nodes: minimax calls searched for the root, the root included (may be NULL).
 * depth: uint8 [n], 0 .. BZ_MINIMAX_MAX_DEPTH; a root with a larger depth is a bounds-check failure (BZ_CHECK) and is
 * not searched (action 255, value 0, nodes 0).  workspace: bz_minimax_workspace_bytes(n) bytes, 16-byte aligned.  The
 * search is alpha-beta, split at the root (one full-window search per root move); every result equals plain minimax.
 * BZ_ERR_ARG: size not 4 / 6 / 8, n < 0 or n >= 2^25, a NULL pointer other than nodes; BZ_ERR_UNALIGNED: workspace. */
#define BZ_MINIMAX_MAX_DEPTH 8
int bz_minimax_moves(const uint64_t *me, const uint64_t *opp, const uint8_t *depth, const uint64_t *key, uint64_t seed,
                     int64_t n, int size, void *workspace, uint8_t *action, int8_t *value, int64_t *nodes,
                     bz_stream_t stream);
int64_t bz_minimax_workspace_bytes(int64_t n);

/* ------------------------------------------------------------------------------------------
 * Exact endgame solver: the perfect player (the definition is oracle/endgame_ref.py; DESIGN.md section 2).  For
 * every mover-relative root i (me[i], opp[i]) with e = size^2 - popcount(me | opp) <= BZ_SOLVE_MAX_EMPTIES empties:
 *  - value(node): if the mover has a legal move, the maximum over its moves of -value(child); else, if the opponent has
 *    one (a pass, reversi_terminal.py:31-35), -value(node with the sides swapped); else (game over)
 *    popcount(me) - popcount(opp), the reference's counts (get_score, reversi_board.py:67-85): empty squares go to nobody.
 *  - value[i]: the root's value (int8).  move_value: int8 [n, 65], -value(child) of every legal move; index 64 holds the
 *    value of a forced pass; every action that is not legal holds -128.
 *  - action[i]: the first maximum of move_value in cell order (the reference's strict ">"), 64 when the mover must pass,
 *    255 when the game is over.
 *  - nodes (may be NULL): positions entered for the root, the root and the positions after passes included.
 * A root with more empties than BZ_SOLVE_MAX_EMPTIES is a bounds-check failure (BZ_CHECK) and is not searched: action
 * 255, value 0, every move value -128, nodes 0.  workspace: bz_endgame_workspace_bytes(n) bytes, 16-byte aligned.  The
 * search is alpha-beta with the full window, split at two plies (one search per root move and reply); every result
 * but nodes equals plain negamax.  BZ_ERR_ARG: size not 4 / 6 / 8, n < 0 or n >= 2^25, a NULL pointer other than
 * nodes; BZ_ERR_UNALIGNED: workspace. */
#define BZ_SOLVE_MAX_EMPTIES 20
int bz_endgame_solve(const uint64_t *me, const uint64_t *opp, int64_t n, int size, void *workspace, uint8_t *action,
                     int8_t *value, int8_t *move_value, int64_t *nodes, bz_stream_t stream);
int64_t bz_endgame_workspace_bytes(int64_t n);

/* Philox4x32-10 of (seed, game_id, ply): the u32 the move sampler draws (for tests). */
int bz_philox_u32(uint64_t seed, const int64_t *game_id, const int32_t *ply, uint32_t *out, int64_t n,
                  bz_stream_t stream);

/* Replay augmentation ("next" row 1 of SURVEY.md section 8f): the 8 dihedral transforms of the
 * reference's dataset expansion (src/tic_tac_toe/SL/train.py:27-36) applied to (board, pi)
 * records: sym[i] in 0..7 = identity, flip rows, flip columns, rot90 x1, x2, x3 (counter-clockwise,
 * torch.rot90), transpose, anti-transpose (the reference's 8th lambda, flip(0).t(), duplicates
 * rot90 x3 and is removed by its dedup; the intended "other diagonal" is used here).  pi: float32
 * [n, 65], the pass entry is invariant.  size in {4, 6, 8}. */
int bz_reversi_symmetry(const uint64_t *me, const uint64_t *opp, const float *pi, const uint8_t *sym,
                        uint64_t *me_out, uint64_t *opp_out, float *pi_out, int64_t n, int size,
                        bz_stream_t stream);

/* 64-bit content hash of every (board, pi) record (me, opp, float32 pi[65]; -0 hashes like +0): the dedup key of the
 * dataset expansion -- the reference keeps the first occurrence of every distinct (state, action) pair of its 8-fold
 * expanded dataset (src/tic_tac_toe/SL/train.py:38-50, a string set); betazero_b200.train.expand_with_transforms sorts
 * by this key and compares the records themselves, so a hash collision cannot merge two different records. */
int bz_record_hash(const uint64_t *me, const uint64_t *opp, const float *pi, uint64_t *hash_out, int64_t n, bz_stream_t stream);

/* Fused policy/value MLP inference (the network is the only dense contraction on the path and the
 * only tensor-core user): x bf16 [n, 128] canonical planes -> 128 -> 256 -> 256 -> 256 (ReLU) ->
 * head, all four layers in ONE tcgen05/TMEM kernel launch.  Architecture = the reference's TicTacToeNet
 * family (src/tic_tac_toe/SL/neural_networks.py:4-30, hidden 256 per SL/train.py:186) widened to
 * 8x8 with a value column.  out: bf16 [n, 72] (65 policy logits, the pre-tanh value, zero padding) =
 * the BZ_PRIOR_LOGITS_BF16 input of bz_mcts_step.  Only this shape is supported.
 *
 * The kernels run on CTA pairs (clusters of 2, tcgen05.mma.cta_group::2): each pair owns 128 rows, each
 * CTA 64 of them and HALF of every weight matrix (the B operand of a pair MMA is split by output row), so
 * the whole net (180 KB per CTA) is resident in shared memory after five bulk copies issued at kernel
 * start.  weight_image_pair: bz_mlp_pair_image_bytes() bytes = [2 ranks][W1 half: 2 K slabs x 128 rows |
 * W2 half: 4 x 128 | W3 half: 4 x 128 | head half: 4 x 40 rows, 128 B per row, K-major SWIZZLE_128B |
 * biases float32 [256 + 256 + 256 + 80]] (betazero_b200.net.pack_mlp_pair_image builds it from the
 * torch.nn.Linear weights; rank r holds rows r*128.. of the hidden layers and rows r*40.. of the 80-row
 * head; both ranks carry all biases).  x, weight_image_pair and out must be 16-byte aligned.
 * (Round 1 also shipped three one-CTA-per-tile variants; they were slower at every batch size and now live,
 * unbuilt, in profiles/experiments/mlp_onecta.cu.) */
int bz_mlp_forward_pair(const void *x_bf16, const void *weight_image_pair, void *out_bf16, int64_t n,
                        bz_stream_t stream);
int64_t bz_mlp_pair_image_bytes(void);
/* The pair kernel for 9 473 .. 18 944 rows: every pair owns TWO 128-row tiles and ping-pongs them (a control warp
 * issues the MMAs of one tile while the 16 epilogue warps convert the other), so 16 384 rows are one wave of 128 CTAs
 * and the tensor cores do not idle during the epilogues; the two 64 KB weight regions of a CTA are recycled layer by
 * layer.  Same weight image, x / out and results as bz_mlp_forward_pair. */
int bz_mlp_forward_pair2(const void *x_bf16, const void *weight_image_pair, void *out_bf16, int64_t n,
                         bz_stream_t stream);

/* INT32 issue-rate microbenchmark for the env roofline denominators.
 * variant 0: SHF + LOP3 chains, all on the ALU pipe (how 64-bit shifts/masks normally compile);
 * variant 1: the same 64-bit shift+mask work with shifts as IMAD (FMA pipe) and masks as LOP3 (ALU pipe).
 * sink: device uint32 [1].  *ops_per_thread (host) receives the integer instructions per thread. */
int bz_int32_microbench(uint32_t *sink, int blocks, int threads, int iters, int variant, int64_t *ops_per_thread,
                        bz_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BETAZERO_B200_H */
