/*
 * az_engine.h — C ABI of the B200-native AlphaZero self-play engine (Connect4).
 *
 * This is the drop-in boundary for the self-play / episode-generation path of
 * pierreveron/alphazero-implementation.  The reference has no FFI layer of its
 * own (it is pure Python); each entry point below names the reference code it
 * replaces (paths relative to src/alphazero_implementation/ of the reference).
 * The Python adapters in alphazero-implementation_b200/ bind these with ctypes
 * and present the reference's class surfaces (EpisodeGenerator, AlphaZeroSearch,
 * Node, Model.predict, Config/State/Action).  See INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 on success, a negative AZ_E_* code on failure;
 *     az_last_error() gives the message.  Nothing throws across the boundary.
 *   - all buffer arguments are DEVICE pointers on the engine's GPU unless the
 *     name ends in _host; sizes are in elements.  The engine owns its arenas;
 *     caller buffers are borrowed for the duration of the call's stream work.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *     Calls only enqueue work unless documented as synchronising.
 *   - boards are two u64 bitboards (stones of player 0 / player 1), bit index =
 *     column*7 + row, row 0 = bottom (the reference's `State.grid[row][col]`,
 *     notebooks/policy_comparison.ipynb#cell6 "Row 0 (bottom)").
 *   - children of a node are ordered by ascending column (`state.actions` order,
 *     models/games/connect4/model.py:29); per-column outputs use column index.
 *   - there is no CPU fallback: az_create fails if no sm_100 device is usable.
 */
#ifndef AZ_ENGINE_H
#define AZ_ENGINE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZ_ABI_VERSION 1

/* status codes */
#define AZ_OK 0
#define AZ_E_INVALID (-1)   /* bad argument / configuration */
#define AZ_E_CUDA (-2)      /* CUDA runtime error (message has the detail) */
#define AZ_E_NOMEM (-3)     /* device allocation failed */
#define AZ_E_STATE (-4)     /* call not valid in the engine's current state */
#define AZ_E_OVERFLOW (-5)  /* an output buffer / episode ring was too small */

/* built-in deterministic evaluators for az_run_simulations (normative definition:
 * oracle/evaluators.py; restated in csrc/az_eval.cuh) */
#define AZ_EVAL_UNIFORM 1 /* prior = fp32(1)/fp32(k) on the k legal columns, value [0,0] */
#define AZ_EVAL_HASH 2    /* priors / value from a 64-bit hash of the position */

/* layouts for az_gather_leaves */
#define AZ_LAYOUT_GRID_F32 0        /* [E,6,7] f32, -1 empty / 0 / 1 owner  (BasicNN._states_to_tensor, basic.py:41-47) */
#define AZ_LAYOUT_PLANES_F32 1      /* [E,3,6,7] f32: empty, side-to-move, opponent (CNNModel._states_to_tensor, cnn.py:77-100) */
#define AZ_LAYOUT_PLANES_BF16 2     /* same planes, bf16 NCHW */
#define AZ_LAYOUT_PLANES_BF16_NHWC 3 /* [E,6,7,8] bf16 channels-last, channels 3..7 zero (tensor-core conv input) */

/* Operand formats of the tensor-core evaluators.  Both are 16-bit operands with fp32 accumulation at the same tcgen05 rate;
 * fp16 carries 11 significand bits against bf16's 8 and is the mode that meets north_star's 1e-3 tolerance against the fp32
 * `predict` (models/games/connect4/model.py:19-43); bf16 is the default BASELINE config 3 names. */
#define AZ_FMT_BF16 0
#define AZ_FMT_F16 1

/* policy_kind for az_expand_backup */
#define AZ_POLICY_LOGITS 0 /* raw logits[E,7]; legal-only fp32 softmax applied (model.py:29-38) */
#define AZ_POLICY_PRIORS 1 /* priors[E,7] already normalised over the legal columns */

/* leaf status written by az_select_leaves */
#define AZ_LEAF_EVAL 0     /* non-terminal leaf waiting for the evaluator */
#define AZ_LEAF_TERMINAL 1 /* terminal leaf, already backed up (search.py:75-77) */
#define AZ_LEAF_IDLE 2     /* slot inactive or in error */
#define AZ_LEAF_SERVED 3   /* non-terminal leaf whose outputs come from the evaluation cache (az_set_eval_cache), not from
                              a row of its own: it is not in the evaluator's list, and expand + backup treat it like AZ_LEAF_EVAL */

/* per-tree error flags (az_root_stats `err`) */
#define AZ_TREE_OK 0
#define AZ_TREE_ROOT_ENDED 3 /* search asked on a finished position: the reference raises AttributeError (search.py:76, parent is None) */

typedef struct az_config {
    int32_t height;          /* 6 */
    int32_t width;           /* 7 */
    int32_t count;           /* 4  (Config(6,7,4), scripts/train.py:12) */
    int32_t num_games;       /* E: concurrent game slots / trees (EpisodeGenerator num_episodes) */
    int32_t num_simulations; /* S: arena is sized for 1 + 7*S nodes per tree (search.py:15) */
    int32_t device;          /* CUDA device ordinal */
    int32_t lanes_per_tree;  /* 32 = one warp per tree, 16 = two, 8 = four trees per warp; 0 = default (8) */
    int32_t hot_nodes_plus1; /* tuning: 0 = automatic; k+1 = keep the first k nodes of every tree in shared memory in az_run_simulations */
    double c_puct;           /* exploration_weight (search.py:16) */
} az_config;

typedef struct az_engine az_engine;

/* counters returned by az_get_stats (totals since az_create / az_reset_stats) */
typedef struct az_stats {
    uint64_t simulations;      /* iterations of search.py:66 summed over trees */
    uint64_t evaluations;      /* non-terminal leaves (one evaluator row each) */
    uint64_t levels;           /* select_child calls (search.py:27) */
    uint64_t children_created; /* add_child calls (node.py:44) */
    uint64_t backup_nodes;     /* nodes touched by backpropagate (search.py:48) */
    uint64_t moves;            /* select_next_node calls (node.py:31) */
    uint64_t episodes;         /* finished games */
    uint64_t children_scanned; /* child records read by select_child (sum of legal moves over levels) */
} az_stats;

int32_t az_abi_version(void);
/* message of the last failure on `h` (or of the last failed az_create when h == NULL) */
const char *az_last_error(const az_engine *h);

/* lifetime.  Replaces: AlphaZeroSearch.__init__ (search.py:11-20) + the Python object heap of Nodes. */
int32_t az_create(const az_config *cfg, az_engine **out);
int32_t az_destroy(az_engine *h);
/* bytes of device memory the engine allocated */
int64_t az_device_bytes(const az_engine *h);
/* CUDA device ordinal the engine lives on */
int32_t az_device(const az_engine *h);

/* ---- game rules (stand-alone; replaces third-party simulator.game.connect, SURVEY App. B) ---- */
/* Action.sample_next_state() (search.py:89, node.py:38) on n boards, plus the successor's
 * State.actions mask / has_ended / reward.  status[i] = 0 ok, 1 illegal (column full, >= width, or game over). */
int32_t az_env_step(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player,
                    const uint8_t *col, int64_t n, uint64_t *out_bb0, uint64_t *out_bb1, uint8_t *out_player,
                    uint8_t *out_legal, uint8_t *out_ended, int8_t *out_reward /*[n][2]*/, uint8_t *out_status,
                    void *stream);
/* State.actions (7-bit mask) / State.has_ended / State.reward of arbitrary positions */
int32_t az_state_info(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int64_t n,
                      uint8_t *out_legal, uint8_t *out_ended, int8_t *out_reward /*[n][2]*/, void *stream);
/* legal-only softmax epilogue of Connect4Model.predict (model.py:26-39): priors[n,7] (0 on illegal columns) */
int32_t az_masked_softmax(az_engine *h, const float *logits /*[n][7]*/, const uint8_t *legal, int64_t n,
                          float *out_priors /*[n][7]*/, void *stream);
/* plane encoders on arbitrary positions (basic.py:41-47, cnn.py:77-100); layout = AZ_LAYOUT_* */
int32_t az_encode_states(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int64_t n,
                         void *out, int32_t layout, void *stream);

/* ---- roots ---- */
/* all E slots to the given initial state with empty trees and empty episode logs
 * (episode_generator.py:42-45).  Resets the move-step counter and the episode ring. */
int32_t az_reset_games(az_engine *h, uint64_t init_bb0, uint64_t init_bb1, int32_t init_player, void *stream);
/* slots 0..n-1 take the given root positions (Node(state), node.py:8), n <= num_games becomes the
 * active tree count for the search calls below.  Does not touch the episode logs. */
int32_t az_set_roots(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int32_t n,
                     void *stream);

/* ---- search ---- */
/* AlphaZeroSearch.run_simulations (search.py:65-91) with a built-in evaluator, all `num_sims`
 * simulations of every active tree in ONE launch (select -> evaluate -> expand -> backup). */
int32_t az_run_simulations(az_engine *h, int32_t num_sims, int32_t eval_kind, void *stream);
/* one simulation step with an external evaluator (the policy/value net), split at the
 * device boundary of search.py:82-84:
 *   az_select_leaves : search.py:69-79  (PUCT descent; terminal leaves are backed up here)
 *   az_gather_leaves : Model._states_to_tensor of the leaves into one packed batch, row i = slot i
 *                      (rows of AZ_LEAF_TERMINAL / AZ_LEAF_IDLE slots are zero-filled)
 *   az_expand_backup : search.py:87-91  (legal-only softmax, add_child x k, backpropagate value[leaf.player]) */
int32_t az_select_leaves(az_engine *h, void *stream);
int32_t az_gather_leaves(az_engine *h, void *out, int32_t layout, void *stream);
int32_t az_expand_backup(az_engine *h, const float *policy /*[E][7]*/, const float *values /*[E][2]*/,
                         int32_t policy_kind, void *stream);
/* az_expand_backup followed by az_select_leaves in one launch (same results): the only tree kernel between two evaluator
 * calls of the simulation loop (search.py:66-91). */
int32_t az_expand_backup_select(az_engine *h, const float *policy, const float *values, int32_t policy_kind, void *stream);
/* the leaves chosen by the last az_select_leaves (for evaluators that want positions, not planes); with symmetric evaluation on
 * (az_set_symmetric_eval), every non-terminal leaf in its canonical orientation and the legal mask of that orientation */
int32_t az_leaf_info(az_engine *h, uint64_t *out_bb0, uint64_t *out_bb1, uint8_t *out_player, uint8_t *out_legal,
                     uint8_t *out_status, void *stream);

/* engine-owned device arrays describing the leaves of the last az_select_leaves (borrowed; valid until az_destroy):
 * lets another kernel consume the leaves without a gather launch (see az_mlp_forward_leaves).  With symmetric evaluation on,
 * non-terminal leaves are in their canonical orientation (az_leaf_mirror tells which were mirrored). */
int32_t az_leaf_arrays(az_engine *h, const uint64_t **bb0, const uint64_t **bb1, const uint8_t **status, int32_t *n_active);
int32_t az_leaf_players(az_engine *h, const uint8_t **player);
/* Leaf compaction.  Terminal leaves (search.py:75-77, ~15 % of the simulations of a running self-play loop) need no evaluation.
 * az_set_leaf_compaction(h, 1): every az_select_leaves / az_expand_backup_select is followed by one more small launch that writes
 * the ordered list of the slots whose leaf waits for the evaluator (status AZ_LEAF_EVAL) and its length; the ResNet evaluators
 * then walk that list and scatter their outputs to the slots' rows.  az_leaf_compact returns the two DEVICE pointers, or NULLs
 * when the last selection ran without compaction (the evaluators then compute every slot's row, zeros for the others).
 * az_set_leaf_compaction(h, 2): az_expand_backup_select builds the list itself (no extra launch): the same slots in the order the
 * warps finished their selections, not ascending - for consumers that scatter per slot, as all evaluators of this library do;
 * az_select_leaves (once per search) still takes the extra launch. */
int32_t az_set_leaf_compaction(az_engine *h, int32_t on);
int32_t az_leaf_compact(az_engine *h, const int32_t **eval_list, const int32_t **eval_count);

/* Evaluation cache of the network-in-the-loop path: an open-addressed table in HBM (2-entry buckets of one 128-byte line)
 * keyed by (position, side to move, weights epoch) that holds the evaluator's 9 outputs (7 logits, 2 values) exactly as it
 * wrote them.  Only for evaluators whose output row is a pure function of the position (deterministic and independent of the
 * batch it falls in): the search then computes the same bits with fewer evaluator rows.  Each selection probes the table for
 * every non-terminal leaf: a published entry serves the leaf (AZ_LEAF_SERVED, no row), a position another tree of the same
 * selection already claimed reuses that tree's row, and otherwise the leaf claims an entry and is evaluated; its expansion
 * publishes the row.  Active while leaf compaction is on (az_set_leaf_compaction 1 or 2).
 * az_set_eval_cache: 2^log2_entries entries of 64 bytes (10 <= log2_entries <= 30), 0 = off; a new size starts an empty table.
 * Call it before capturing a CUDA graph of the search: launches bake the table's address in. */
int32_t az_set_eval_cache(az_engine *h, int32_t log2_entries);
/* Entries written before this call stop matching (a device word, so captured graphs see it): call it whenever the evaluator's
 * weights change in place or another evaluator takes over. */
int32_t az_bump_eval_epoch(az_engine *h, void *stream);
typedef struct az_eval_cache_stats {
    uint64_t rows;          /* non-terminal leaves the evaluator computed a row for */
    uint64_t hits;          /* leaves served from a published entry */
    uint64_t followers;     /* leaves that reused the row of another tree's leaf in the same selection */
    uint64_t failed_claims; /* leaves evaluated without caching: no entry of their bucket could be claimed */
    uint64_t evictions;     /* published entries of the current epoch replaced by a claim */
} az_eval_cache_stats;
/* totals since az_create / az_reset_stats (az_stats.evaluations = rows + hits + followers).  Synchronises. */
int32_t az_get_eval_cache_stats(az_engine *h, az_eval_cache_stats *out_host, void *stream);

/* ---- left-right mirror symmetry of Connect4 (off by default; with it off every result is unchanged) ----
 * mirror(b) moves column c's 7 bits (bit 7c + r) to column 6 - c, in both bitboards; the side to move does not change.  The
 * canonical form of a position is the smaller of it and its mirror, comparing (bb0, bb1) as unsigned 64-bit values, bb0 first;
 * a palindrome (its own mirror) is its own canonical form and is not mirrored.
 * az_set_symmetric_eval(h, 1): the network-in-the-loop search evaluates f_sym(x) = f(canon(x)) with the policy columns reversed
 * when canon(x) is the mirror of x.  Each selection writes the canonical form of every non-terminal leaf to the leaf arrays (what
 * az_gather_leaves, az_leaf_info, az_leaf_arrays and every evaluator read) and probes the evaluation cache with it; the expansion
 * stores canonical column c's prior at actual column 6 - c of a mirrored leaf.  The tree, root statistics, root noise and the
 * episode ring stay in the actual orientation.  f_sym is a pure function of the position, so the cache stays exact; its entries
 * hold plain rows f(y) keyed by y and stay valid when the mode changes.  Adds no launch.  AZ_E_STATE while a selection's leaves
 * wait for their expansion; call it before capturing a CUDA graph of the search (launches bake the kernel choice in).  The fused
 * built-in path (az_run_simulations, az_run_move_step) has no symmetric variant: it returns AZ_E_STATE while the mode is on. */
int32_t az_set_symmetric_eval(az_engine *h, int32_t on);
/* [E] u8 device array (borrowed; valid until az_destroy): 1 where the last selection's leaf is the mirror of the position the
 * descent reached (0 for palindromes, terminal and idle slots); NULL when the last selection ran with the mode off */
int32_t az_leaf_mirror(az_engine *h, const uint8_t **mirrored);
/* out = mirror(in) for the n positions (device arrays), or, with flags (u8 [n], may be NULL = every row), only for the rows
 * whose flag is non-zero (the others are copied).  The output may be the input. */
int32_t az_mirror_states(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *flags, int64_t n, uint64_t *out_bb0,
                         uint64_t *out_bb1, void *stream);

/* ---- results ---- */
/* root statistics of every active tree, per column (0 on illegal columns):
 * child visit counts (Node.improved_policy = child_N / (root_N - 1), node.py:23-29), child value sums,
 * child priors, root value_sum / visit_count (Node.value, node.py:50-55), legal mask, AZ_TREE_* flag.
 * Any output pointer may be NULL. */
int32_t az_root_stats(az_engine *h, int32_t *child_N /*[n][7]*/, double *child_W /*[n][7]*/,
                      float *child_P /*[n][7]*/, double *root_W, int32_t *root_N, uint8_t *legal, int32_t *err,
                      void *stream);
/* the whole SoA tree of one slot (value_sum f64, visit_count u32, prior f32, first-child index u32;
 * node 0 = root, 0 = no children).  Buffers hold az_tree_capacity() entries.  Synchronises. */
int32_t az_tree_capacity(const az_engine *h);
int32_t az_export_tree(az_engine *h, int32_t slot, double *W, uint32_t *N, float *P, uint32_t *first_child,
                       int32_t *used_host);

/* ---- self-play (episode_generator.py:53-78) ---- */
/* For every slot in slot order semantics: record the sample (root position, child visit counts),
 * draw the move with the supplied uniform exactly as np.random.choice(k, p=N_c/(N-1)) would
 * (node.py:31-35), advance the root (no subtree reuse unless az_set_subtree_reuse, node.py:37-41); if the successor is terminal,
 * finish the episode (outcome = successor reward, episode.py:52-54), move it to the episode ring and
 * recycle the slot to the initial state.  finished[slot] (may be NULL) = 1 where an episode finished.
 * Increments the move-step counter. */
int32_t az_sample_moves(az_engine *h, const double *uniforms /*[E]*/, uint8_t *finished, void *stream);
/* One whole move step of the self-play loop (episode_generator.py:53-78) with a built-in deterministic evaluator in ONE
 * launch: az_run_simulations(num_sims, evaluator_kind) followed by az_sample_moves(uniforms, finished), same results.
 * The root's child statistics never leave the registers and the discarded tree is not written back (no subtree reuse unless
 * az_set_subtree_reuse: then it runs as az_run_simulations + az_sample_moves, whose k_reroot keeps the played child's subtree). */
int32_t az_run_move_step(az_engine *h, int32_t num_sims, int32_t evaluator_kind, const double *uniforms /*[E]*/, uint8_t *finished,
                         void *stream);
/* ---- self-play exploration (absent from the reference, which ships DeepMind's pseudocode for them only; both off by default,
 * and with both off every result is the reference's) ---- */
/* Dirichlet noise on the root priors: add_exploration_noise of deepmind_alphazero_pseudocode.py.  A search on fresh roots runs
 * one simulation (which expands a non-terminal root), then az_apply_root_noise, then the remaining S - 1 simulations.  For
 * every active tree whose root has children it draws eta ~ Dirichlet(alpha, ..., alpha) over the k legal columns (ascending;
 * 0 on illegal columns; k = 1 gives 1) and rewrites each root child's prior in place, in fp32 with one rounding per operation:
 *   P' = RN(RN(RN(1 - fraction) * P) + RN(fraction * eta)).
 * eta is a pure function of (seed, slot_offset + slot, number of applications since az_set_root_noise, column): a run is
 * reproduced from its seed, and an engine over slots [lo, hi) with slot_offset = lo draws the rows [lo, hi) of an engine over
 * all slots.  (Philox4x32-10 counters, Marsaglia-Tsang Gamma variates, log space for alpha < 1: see k_root_noise.)
 * az_set_root_noise: alpha in (0, 1e6], fraction in [0, 1], slot_offset >= 0, else AZ_E_INVALID; NULL = off.  Resets the
 * application counter. */
typedef struct az_root_noise {
    double alpha;        /* Dirichlet concentration (pseudocode: root_dirichlet_alpha) */
    float fraction;      /* weight of the noise (pseudocode: root_exploration_fraction) */
    uint64_t seed;
    int64_t slot_offset; /* global index of this engine's slot 0 */
} az_root_noise;
int32_t az_set_root_noise(az_engine *h, const az_root_noise *cfg);
/* the mixing, once per search: valid only after exactly one complete simulation on the current roots (AZ_E_STATE otherwise,
 * and inside a CUDA graph capture).  One k_root_noise launch; increments the application counter. */
int32_t az_apply_root_noise(az_engine *h, void *stream);
/* eta[num_games][7] (device) of the last application (0 for trees it skipped: inactive, in error or without children) */
int32_t az_root_noise_values(az_engine *h, float *eta, void *stream);
/* Temperature cutoff: select_action of deepmind_alphazero_pseudocode.py with num_sampling_moves = plies.  From ply `plies` of a
 * game on, az_sample_moves / az_run_move_step play the most visited root child (the lowest column on ties) instead of sampling
 * node.py:31-35; the uniform of the slot is still an argument and the sample is recorded as before.  Negative = off (default).
 * With the cutoff on, az_run_move_step runs as az_run_simulations + az_sample_moves (two launches, same results). */
int32_t az_set_greedy_from(az_engine *h, int32_t plies);

/* ---- subtree reuse (AlphaGo Zero: the child of the played move becomes the new root and keeps its subtree with all its
 * statistics; off by default, and with it off every result is unchanged) ----
 * Each search still runs num_simulations = S new simulations.  After a move to child c of a root:
 *   - c is expanded and N(c) + S <= max_root_visits (= V): the subtree of c becomes the tree (retained).  Its nodes keep their
 *     relative order, so every children block stays contiguous and in column order; c becomes node 0 with {N(c), W(c), prior 0};
 *   - c was never expanded: a fresh root (N = W = 0, no children);
 *   - N(c) + S > V: a fresh root as well (dropped);
 *   - a game that ended is recycled as before.
 * A subtree of N(c) visits has at most 1 + 7 N(c) nodes, so trees stay within 1 + 7 V nodes and visit counts within V.
 * az_set_subtree_reuse: V = 0 (off, the default) or S <= V <= 65536, else AZ_E_INVALID.  Sizes the arena for 1 + 7 V nodes per tree
 * (az_tree_capacity) and the PUCT tables for counts up to V (AZ_E_NOMEM, and the engine unchanged, if that fails) and resets every
 * tree to a fresh root; root positions and game logs are kept.  V = S never retains a subtree (same results as off).  AZ_E_STATE
 * while a selection's leaves wait for their expansion.  Call it before capturing a CUDA graph of the search: launches bake the
 * arena (tree arrays, tables, capacity) in.  While reuse is on, az_sample_moves runs k_sample_moves then k_reroot, and
 * az_run_move_step runs as az_run_simulations + az_sample_moves. */
int32_t az_set_subtree_reuse(az_engine *h, int32_t max_root_visits);
/* "Play this move, keep the tree": plays cols[t] (u8, device) on every active root under the rule above.  out_status[t] (u8,
 * device) = 0 when played; 1 for an illegal column (or a root in error), which leaves the slot untouched.  A move that ends the game
 * makes that position the root of a fresh tree flagged AZ_TREE_ROOT_ENDED, as az_set_roots would.  Game logs are not touched.
 * AZ_E_STATE while reuse is off or a selection's leaves wait for their expansion. */
int32_t az_advance_roots(az_engine *h, const uint8_t *cols, uint8_t *out_status, void *stream);
typedef struct az_reuse_stats {
    uint64_t retained; /* moves whose played child's subtree was kept */
    uint64_t fresh;    /* moves to a child that was never expanded */
    uint64_t dropped;  /* moves to an expanded child with N(c) + S > V */
    uint64_t nodes;    /* nodes of the retained subtrees */
    uint64_t visits;   /* root visits of the retained subtrees, N(c) */
} az_reuse_stats;
/* totals since az_create / az_reset_stats over moves from a searched root that did not end the game.  Synchronises. */
int32_t az_get_reuse_stats(az_engine *h, az_reuse_stats *out_host, void *stream);

/* Playout cap randomization (KataGo): the searches of the self-play move steps (after az_reset_games and after every
 * az_sample_moves) are each "full" with probability p_full, else "fast".  A full search runs num_simulations new simulations,
 * a fast one fast_sims; a tree that has run its share is idle for the rest of the move step (no leaf, no evaluator row, no cache
 * probe), so a step costs fewer evaluator rows.  Every move is played and logged as before, but a finished game emits only the
 * samples of its full searches, in order: ep_len counts them and may be 0 (the episode is still emitted, with its outcome).
 * Fast searches get no root noise (their η row is 0).
 *   visit_budget = 1 (for subtree reuse): a search tops the root up to num_simulations (fast_sims) visits instead, at least one
 *   new simulation: n = max(S_t - N_start, 1).  With reuse off N_start = 0 and this is the plain cap.
 * The flag of (slot, move step) is a function of (seed, slot_offset + slot, step) alone: Philox4x32-10 keyed by the seed, counter
 * {global slot lo, hi, step, 0xC0000000}, full iff (x + 0.5) / 2^32 < p_full in fp64 - sharded self-play draws what the
 * unsharded run draws.  az_set_roots and az_advance_roots make every search full with S new simulations, visit_budget or not:
 * they are not self-play.  The budgets live in device memory, so a captured simulation graph stays valid from move to move;
 * switching the mode on or off changes the kernels a launch uses (capture after it).  The flags of the game logs apply only while
 * the mode is on: with it off a finished game emits every ply, and switching it on counts every ply already in the logs as full -
 * also a fast ply of an earlier period with the mode on, which its game would have emitted had it ended while the mode was off. */
typedef struct az_playout_cap {
    int32_t fast_sims;     /* new simulations of a fast search, 1 .. num_simulations */
    float p_full;          /* probability of a full search, [0, 1] */
    uint64_t seed;
    int64_t slot_offset;   /* global index of this engine's slot 0, [0, 2^62] */
    int32_t visit_budget;  /* 0 or 1 */
} az_playout_cap;
/* cfg NULL = off (the default).  Draws the flags and budgets of the current roots (synchronises).  AZ_E_INVALID for values out
 * of range, AZ_E_STATE while a selection's leaves wait for their expansion. */
int32_t az_set_playout_cap(az_engine *h, const az_playout_cap *cfg);
/* the current draw: budget[num_games] u32 = the root visit count at which each tree stops (N_start + n), full[num_games] u8;
 * device or pinned host memory, either may be NULL.  AZ_E_STATE before the first az_set_playout_cap. */
int32_t az_search_budgets(az_engine *h, uint32_t *budget, uint8_t *full, void *stream);
typedef struct az_cap_stats {
    uint64_t full_searches;     /* self-play searches that ended in a move, by kind */
    uint64_t fast_searches;
    uint64_t samples_recorded;  /* samples of finished games emitted / left out (fast searches) */
    uint64_t samples_dropped;
    uint64_t simulations;       /* new simulations actually run (az_stats.simulations) */
} az_cap_stats;
/* totals since az_create / az_reset_stats.  Synchronises. */
int32_t az_get_cap_stats(az_engine *h, az_cap_stats *out_host, void *stream);

/* number of finished episodes / samples waiting in the ring.  Synchronises on `stream`. */
int32_t az_episode_counts(az_engine *h, int64_t *n_episodes_host, int64_t *n_samples_host, void *stream);
/* copy the ring out (device buffers sized from az_episode_counts) and empty it.  Episodes appear in
 * ring order; sort by (ep_step, ep_slot) for the reference's yield order.  Synchronises.
 *   ep_*: per episode  — slot, move-step at which it finished, length, first sample index, outcome
 *         (reward of player 0 / player 1: +1 / -1 / 0)
 *   s_* : per sample   — position, side to move, root child visit counts by column */
int32_t az_drain_episodes(az_engine *h, int64_t ep_cap, int64_t s_cap, int32_t *ep_slot, int32_t *ep_step,
                          int32_t *ep_len, int64_t *ep_offset, int8_t *ep_outcome /*[n][2]*/, uint64_t *s_bb0,
                          uint64_t *s_bb1, uint8_t *s_player, int32_t *s_counts /*[n][7]*/,
                          int64_t *n_episodes_host, int64_t *n_samples_host, void *stream);

/* Double-buffered use of the ring (lets the host read one move step's episodes while the next step runs):
 * az_swap_episode_ring makes the other ring the active one (zeroing its counters on `stream`) and reports the
 * index of the ring that was active; that ring keeps its contents until it becomes active again.
 * az_ring_counts synchronises `stream` and returns a ring's counters; az_read_episode_ring enqueues copies of
 * exactly n_episodes / n_samples entries.  Destinations may be device or pinned host memory. */
int32_t az_swap_episode_ring(az_engine *h, int32_t *previous_ring_host, void *stream);
int32_t az_ring_counts(az_engine *h, int32_t ring, int64_t *n_episodes_host, int64_t *n_samples_host, void *stream);
int32_t az_read_episode_ring(az_engine *h, int32_t ring, int64_t n_episodes, int64_t n_samples, int32_t *ep_slot,
                             int32_t *ep_step, int32_t *ep_len, int64_t *ep_offset, int8_t *ep_outcome /*[n][2]*/,
                             uint64_t *s_bb0, uint64_t *s_bb1, uint8_t *s_player, int32_t *s_counts /*[n][7]*/,
                             void *stream);

/* ---- instrumentation ---- */
int32_t az_get_stats(az_engine *h, az_stats *out_host, void *stream); /* synchronises */
int32_t az_reset_stats(az_engine *h, void *stream);
/* checks the table-based fp64 division used by the PUCT score against IEEE division on n pseudo-random
 * (x, d) pairs, d an integer below num_simulations + 2 (max_root_visits + 2 with az_set_subtree_reuse); *mismatches_host must
 * come back 0.  Synchronises. */
int32_t az_selftest_division(az_engine *h, int64_t n, uint64_t seed, int64_t *mismatches_host);
/* number of kernels this engine has launched since az_create */
int64_t az_launch_count(const az_engine *h);

/* ---- fused tensor-core evaluator for the reference's BasicNN (models/games/connect4/basic.py:8-39) ----
 * 42 -> 512 (ReLU) -> 512 (ReLU) -> {7 policy logits, 2 values (tanh)} in ONE kernel: tcgen05.mma (bf16 in, fp32
 * accumulate in tensor memory), bias / ReLU / tanh epilogues in fp32, activations never leave the SM.
 * az_mlp_set_weights takes fp32 DEVICE pointers in nn.Linear layout (weight [out][in]) — the analogue of
 * `inference_model.load_state_dict(model.state_dict())` (search.py:22-25) — and repacks them as bf16 MMA operands.
 * az_mlp_forward consumes the AZ_LAYOUT_GRID_F32 batch written by az_gather_leaves and writes logits [n][7] and
 * values [n][2] in the form az_expand_backup reads. */
typedef struct az_mlp az_mlp;
int32_t az_mlp_create(int32_t device, az_mlp **out);
int32_t az_mlp_destroy(az_mlp *m);
const char *az_mlp_last_error(const az_mlp *m);
/* AZ_FMT_BF16 (default) or AZ_FMT_F16 operands; takes effect at the next az_mlp_set_weights */
int32_t az_mlp_set_operand_format(az_mlp *m, int32_t fmt);
int32_t az_mlp_set_weights(az_mlp *m, const float *w1 /*[512][42]*/, const float *b1, const float *w2 /*[512][512]*/,
                           const float *b2, const float *w_policy /*[7][512]*/, const float *b_policy,
                           const float *w_value /*[2][512]*/, const float *b_value, void *stream);
int32_t az_mlp_forward(az_mlp *m, const float *grid /*[n][42]*/, int64_t n, float *logits /*[n][7]*/,
                       float *values /*[n][2]*/, void *stream);
/* the same with the leaf gather fused in: row i = the leaf of slot i chosen by the last az_select_leaves on `engine` */
int32_t az_mlp_forward_leaves(az_mlp *m, az_engine *engine, float *logits /*[E][7]*/, float *values /*[E][2]*/, void *stream);
int64_t az_mlp_launch_count(const az_mlp *m);

/* ---- fused tensor-core trunk of the ResNet-style net (src/alphazero_simple/resnet.py:13-53, 64 channels, BatchNorm folded) ----
 * stem conv3x3 + num_blocks residual blocks in ONE tcgen05 kernel (csrc/az_conv.cu), the leaf gather fused in;
 * activations stay in shared memory between layers.  Output: [E][6][7][64] bf16 NHWC for the policy / value heads. */
int64_t az_trunk_weight_bytes(int32_t num_blocks);
int32_t az_trunk_forward_leaves(az_engine *engine, const void *packed_weights, const float *biases /*[1+2*num_blocks][64]*/,
                                int32_t num_blocks, void *out, void *stream);
/* trunk + policy / value heads in the same kernel -> logits [E][7], values [E][2] (tanh, [v, -v] as cnn.py:73), the inputs
 * of az_expand_backup.  head_conv_w: 9 taps x [48 out][64 in] bf16 MMA operands (rows 0..31 = policy conv1x1 in the centre tap,
 * rows 32..34 = value conv3x3, BatchNorm folded); head_conv_b [48]; fc_* fp32 in nn.Linear layout ([7][1344], [7], [126], [1]). */
int32_t az_resnet_forward_leaves(az_engine *engine, const void *packed_weights, const float *biases, int32_t num_blocks,
                                 const void *head_conv_w, const float *head_conv_b, const float *fc_policy_w,
                                 const float *fc_policy_b, const float *fc_value_w, const float *fc_value_b, float *logits,
                                 float *values, void *stream);
typedef struct az_resnet_desc {
    int32_t num_blocks;      /* residual blocks (resnet.py:51-53) */
    int32_t num_channels;    /* trunk width: 64, or 128 = the reference's own instance */
    int32_t operand_format;  /* AZ_FMT_*: format of trunk_w / head_conv_w and of the activations between layers */
    int32_t variant;         /* 0: layer-pipelined kernel (csrc/az_resnet_pipe.cu; weights: models.py:pack_trunk_weights_pipe);
                                1: ping-pong kernel, 64 channels only (csrc/az_conv.cu; weights: models.py:pack_trunk_weights);
                                2: variant 0 with two 4-position CTAs per SM, 64 channels, at most 5 blocks;
                                3: variant 2 with CTA pairs (cta_group::2; weights packed as halves, pack_trunk_weights_pipe(pair=True));
                                4: 64 channels, the three taps of a filter row fused into one MMA (N = 192), two tiles ping-pong
                                   (csrc/az_resnet_wide.cu; same packed weights as variant 0) */
    const void *trunk_w;     /* packed 16-bit MMA operands */
    const float *trunk_b;    /* [1 + 2*num_blocks][num_channels] */
    const void *head_conv_w; /* [48 out] x num_channels x 9 taps, packed like trunk_w (models.py:pack_head_weights) */
    const float *head_conv_b;
    const float *fc_policy_w, *fc_policy_b, *fc_value_w, *fc_value_b; /* fp32, nn.Linear layout */
} az_resnet_desc;
int32_t az_resnet_forward_leaves_v2(az_engine *engine, const az_resnet_desc *desc, float *logits, float *values, void *stream);
/* bytes of packed trunk weights the layer-pipelined kernel expects (models.py:pack_trunk_weights_pipe); -1 for an unsupported width */
int64_t az_resnet_pipe_weight_bytes(int32_t num_blocks, int32_t num_channels);
/* ---- CNNModel (models/games/connect4/cnn.py:8-75) on the tensor cores: csrc/az_cnn.cu ----
 * conv3x3 3 -> 64 -> 128 -> 256 (BatchNorm folded, ReLU) in one kernel, Linear 10752 -> 512 + ReLU and both heads in a second;
 * logits [E][7], values [E][2] = [v, -v] (cnn.py:73) for the leaves of the last selection.  Weights are packed by
 * alphazero-implementation_b200/models.py:pack_cnn_weights; `workspace` holds the conv output between the kernels. */
typedef struct az_cnn_desc {
    int32_t operand_format;  /* AZ_FMT_* */
    int32_t reserved;
    const void *conv_w;      /* az_cnn_conv_weight_bytes() bytes */
    const float *conv_b;     /* [64 + 128 + 256] */
    const void *fc_w;        /* az_cnn_fc_weight_bytes() bytes: [336 K chunks][512][32], k = pixel * 256 + channel */
    const float *fc_b;       /* [512] */
    const float *head_w;     /* [8][512] fp32: policy_head.weight rows 0..6, value_head[0].weight row 7 */
    const float *head_b;     /* [8] */
    void *workspace;         /* >= az_cnn_workspace_bytes(num_games) bytes */
    int64_t workspace_bytes;
} az_cnn_desc;
int64_t az_cnn_conv_weight_bytes(void);
int64_t az_cnn_fc_weight_bytes(void);
int64_t az_cnn_workspace_bytes(int64_t n);
int32_t az_cnn_forward_leaves(az_engine *engine, const az_cnn_desc *desc, float *logits, float *values, void *stream);

/* Measurement hook of k_resnet_wide (az_resnet_desc.variant 4): `buf` = device array of 4 + 2 * cap uint64 - [0] launches so far,
 * [1] scratch, then per launch (slot = launch % cap) {first CTA start, last CTA end} on the device's global timer in ns; the caller
 * initialises the pairs to {~0, 0}.  The pointer is baked into launches (and captured graphs) made after the call; NULL = off.
 * bench.py uses it to time the kernel INSIDE the timed region (no reference counterpart). */
int32_t az_resnet_wide_set_timing(void *buf, int32_t cap);

/* Tuning switch of the kernel behind the calls above: 0 (default) = one CTA per 8 positions, 1 = CTA pairs
 * (tcgen05 cta_group::2, M = 256).  Same results; returns the previous setting. */
int32_t az_trunk_set_cta_pair(int32_t on);

#ifdef __cplusplus
}
#endif
#endif /* AZ_ENGINE_H */
