// B200-native AlphaZero self-play engine: MCTS tree arena + Connect4 rules + leaf gather.
// C ABI in include/az_engine.h.  Built for sm_100a only; there is no CPU path.
//
// Data layout in HBM (structure of arrays, tree-major, `cap` = roundup8(1 + 7*S) nodes per tree, 1 + 7*V with subtree reuse):
//   W[E][cap] f64     value_sum (node.py:14); fp64 because the reference sums Python floats
//   M[E][cap] uint4   {visit_count u32 (node.py:13), prior f32 bits (node.py:15), first-child index u32, 0}
//                     one 16-byte vector load per child; children of a node are contiguous in ascending
//                     column order (= dict insertion order of node.children, search.py:88-90); 0 = not expanded
// Node 0 is the root.  Positions are NOT stored per node: the descent replays the chosen columns on the
// root bitboards held in registers (a drop + line test is ~20 integer ops; a node-sized load is not).
//
// Work decomposition: eight lanes own one tree for the whole launch (TPW = 4 trees per warp), or a whole
// warp owns one (TPW = 1; its four 8-lane quarters then compute the same thing).  Lane c (< 7) of each
// quarter handles column c of the current node: it loads that child's record (coalesced: neighbouring
// lanes read neighbouring records), scores it in fp64 with the reference's operation order and
// rounding, and the best child is found with a __shfl_xor butterfly (lowest column among the maxima =
// the reference's strict '>' first-maximum rule).  The warp stays converged and the level loop and the
// per-simulation tail are straight-line code: lanes of finished trees compute on stale valid values and
// every state update is masked, so every shuffle / ballot uses the full mask and no reconvergence
// barrier sits on the dependent chain.  A tree is owned by one quarter, so updates need no atomics;
// __syncwarp orders them between lanes.
//
// A simulation is one long dependent chain (with thousands, not millions, of trees nothing else hides
// it), so the kernels are organised around that chain: see descend(), k_run_sims and DESIGN.md section 3.
// The fused kernel keeps the first ~400 nodes of every tree (16-byte HotNode records) and the 1/d, sqrt
// tables in shared memory, the root's statistics in registers, and can append the self-play move
// (az_run_move_step); the split path (k_select / k_expand_backup / k_expand_select) serves external
// evaluators and issues every independent load in its first round.
//
// fp64 without the division subroutine: the divisors of PUCT are small integers (visit counts <= S),
// so 1/d and sqrt(n) come from tables of correctly rounded values (built once per engine with
// __drcp_rn / __dsqrt_rn) and x/d is finished with two FMA residual corrections, which yields the
// correctly rounded quotient (Markstein); tests/test_gpu_search.py checks it against __ddiv_rn.
#include <assert.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <cuda_bf16.h>

#include "../../include/az_engine.h"
#include "az_eval.cuh"
#include "c4_bitboard.cuh"

namespace {

constexpr int PATH_STRIDE = 44;  // root + at most 42 plies (+1 pad)
constexpr int MAX_PLIES = 42;
constexpr int NSTAT = 11;  // per-tree counters: sims, evals, levels, children, moves, episodes, children scanned, then the evaluation
                           // cache's hits, followers, failed claims, evictions
constexpr unsigned FULL = 0xFFFFFFFFu;

// One entry of the evaluation cache (az_set_eval_cache), two per 128-byte bucket.  `ctrl` is the entry's state word: kind in
// bits 0-1, the selection launch that set it in bits 2-31, a slot in bits 32-63.  Key, tag and payload are written only while
// the entry is BUSY (taken by a CAS on ctrl), so a reader that sees the same non-BUSY ctrl before and after reading them holds
// a consistent copy (a seqlock); ctrl never returns to an earlier value, because a slot claims or publishes at most once per launch.
struct __align__(64) CacheEntry {
    float4 p0, p1;  // outputs 0..7 as the evaluator wrote them: logits 0..6, value 0
    float v1;       // output 8: value 1
    uint32_t tag;   // weights epoch * 2 + side to move
    unsigned long long ctrl;
    unsigned long long b0, b1;  // the position
};
static_assert(sizeof(CacheEntry) == 64, "two entries per 128-byte bucket");

struct Arena {
    double *W;
    uint4 *M;  // x = N, y = prior bits, z = first child, w = 0
    const double *rcp;  // rcp[d] = RN(1/d), d = 0 .. S+1 (rcp[0] unused)
    const double *sqt;  // sqt[n] = RN(sqrt(n))
    const double2 *t2;  // t2[n] = {rcp[n + 1], sqt[n]}: what a child with n visits contributes to a level, in one 16-byte load
    uint64_t *root_bb0, *root_bb1;
    uint8_t *root_player;
    uint32_t *used;
    int32_t *tree_err;
    // leaves of the split (external evaluator) path
    uint32_t *leaf_node;
    uint64_t *leaf_bb0, *leaf_bb1;
    uint8_t *leaf_player, *leaf_status, *leaf_depth;
    uint32_t *path;    // [E][PATH_STRIDE]
    uint32_t *tstats;  // [E][NSTAT]
    int32_t *eval_list;   // [E] slots whose leaf waits for the evaluator: ascending (k_compact_leaves) or in ticket order (k_expand_select<COMPACT>)
    int32_t *eval_count;  // [4] [0] = entries in eval_list; [2..3] one 64-bit word: tickets | warps through << 32 (k_expand_select<COMPACT>; zero between launches)
    // evaluation cache (az_set_eval_cache; the kernels that use it are the CACHE instantiations)
    CacheEntry *cache;         // [2 * (cache_mask + 1)]: buckets of two entries
    uint32_t cache_mask;       // buckets - 1
    uint32_t *cache_ctl;       // [0] selection launches so far (advanced once after each selection launch), [1] weights epoch
    uint32_t *leaf_src;        // [E] row the leaf's outputs come from: the slot itself, the leader slot of a follower, or SRC_HIT
    uint32_t *leaf_claim;      // [E] entry the leaf claimed (its expansion publishes the row there), NO_CLAIM if none
    float4 *cached_out;        // [E][3] the 9 outputs of a leaf served by a hit
    // game in progress per slot
    uint64_t *g_bb0, *g_bb1;  // [E][42]
    uint8_t *g_player;        // [E][42]
    int32_t *g_counts;        // [E][42][7]
    int32_t *g_len;           // [E]
    // finished-episode ring
    unsigned long long *ring;  // [0] episodes, [1] samples, [2] dropped
    int32_t *ep_slot, *ep_step, *ep_len;
    int64_t *ep_offset;
    int8_t *ep_outcome;  // [cap][2]
    uint64_t *s_bb0, *s_bb1;
    uint8_t *s_player;
    int32_t *s_counts;  // [cap][7]
    int64_t ep_cap, s_cap;
    int cap;  // nodes per tree
    int E;
    int tab_n;  // entries in rcp / sqt
};

// ------------------------------------------------------------------------------------------------
// exact fp64 helpers
// x / d for an integer 1 <= d < tab_n, correctly rounded: r = RN(1/d) from the table, then two
// residual corrections (q += (x - d*q) * r).  The first makes q faithful, the second exact-rounded.
__device__ __forceinline__ double div_tab(double x, uint32_t d, const double *__restrict__ rcp) {
#ifdef AZ_DEBUG_BOUNDS
    assert(d < 1u << 20);  // tables hold num_simulations + 8 entries; a wild index shows up here first
#endif
    const double r = rcp[d];  // generic load: the tables live in shared memory (fused kernel, small S) or in global memory
    const double nd = -(double)d;
    double q = __dmul_rn(x, r);
    q = __fma_rn(__fma_rn(nd, q, x), r, q);
    return __fma_rn(__fma_rn(nd, q, x), r, q);
}

// score = child.value + c * child.prior * sqrt(node.visit_count) / (1 + child.visit_count), evaluated
// left to right in fp64 with one rounding per operation (search.py:33-40).  child.value = W/N, 0 if N == 0
// (node.py:50-55); W == 0 gives q = 0 without dividing (N == 0 implies W == 0).
__device__ __forceinline__ double puct_score(uint32_t n, double w, float p, double sq, double c_puct,
                                             const double *__restrict__ rcp) {
    const double u = div_tab(__dmul_rn(__dmul_rn(c_puct, (double)p), sq), 1u + n, rcp);
    const double q = (w == 0.0) ? 0.0 : div_tab(w, n, rcp);
    return __dadd_rn(q, u);
}

struct Child {  // the record of "my" column's child at the current node
    double w;
    double sq;  // sqrt(n): the sqrt(node.visit_count) of the NEXT level if this child is selected, fetched ahead of the need
    double r1, r0;  // RN(1/(1+n)), RN(1/n): the two reciprocals of this child's PUCT score (latency variant only)
    double x;       // (c * prior) * sqrt(N_parent): the numerator of U, computed while the table entries are in flight (latency variant)
    double d1, d0;  // 1 + n, n as doubles (the divisions' residual steps), converted ahead of the need (latency variant)
    uint32_t n, cb;
    float p;
};

// The tables a kernel reads, in whatever memory they live (shared memory in the fused kernel when they fit, else global).
struct Tabs {
    const double *rcp;   // rcp[d]
    const double2 *t2;   // {rcp[n + 1], sqt[n]}
};

// x / d with the reciprocal r = RN(1/d) and d as a double already in registers (same arithmetic as div_tab)
__device__ __forceinline__ double div_r(double x, double d, double r) {
    const double nd = -d;  // folds into the FMA's operand modifier
    double q = __dmul_rn(x, r);
    q = __fma_rn(__fma_rn(nd, q, x), r, q);
    return __fma_rn(__fma_rn(nd, q, x), r, q);
}

// puct_score with everything but the two divisions done when the child record arrived (load_child): the numerator
// x = (c * P) * sqrt(N), both reciprocals and both divisors as doubles
__device__ __forceinline__ double puct_score_pre(const Child &ch) {
    const double u = div_r(ch.x, ch.d1, ch.r1);
    const double q = (ch.w == 0.0) ? 0.0 : div_r(ch.w, ch.d0, ch.r0);
    return __dadd_rn(q, u);
}

// first maximum over the 7 columns of an 8-lane quarter: a butterfly over (score, column) pairs - the larger score wins,
// equal scores keep the lower column (the reference's strict `>` scan keeps the first maximum).  Every lane of the
// quarter ends with the same column.  (Carrying the column costs one extra shuffle per round, issued alongside the
// score's two, and saves the equality ballot + find-first-set that would follow a plain max.)
// The score's own chain is shuffle -> compare -> select per round (on a tie either operand is the same value); the tie-break
// only steers the column, whose chain is shuffle -> select with the predicates already computed - two chained fp64 compares
// per round are off the score's path.
__device__ __forceinline__ int argmax_first(double score, int c) {
    double m = score;
    int mi = c;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) {
        const double o = __shfl_xor_sync(FULL, m, off);
        const int oi = __shfl_xor_sync(FULL, mi, off);
        const bool gt = o > m;
        const bool take = gt || (o == m && oi < mi);
        m = gt ? o : m;
        mi = take ? oi : mi;
    }
    return mi;
}

// Throughput variant of the same selection: plain max butterfly (two shuffles per round), then the lowest lane holding the
// maximum by ballot + find-first-set.  Four shuffles fewer per level; the ballot / ffs tail is longer on the dependent chain.
__device__ __forceinline__ int argmax_first_ballot(double score, int sub) {
    double m = score;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) {
        const double o = __shfl_xor_sync(FULL, m, off);
        m = (o > m) ? o : m;
    }
    const unsigned eq = __ballot_sync(FULL, score == m);
    return __ffs((eq >> sub) & 0xFFu) - 1;
}


// One tree's node storage as seen by a kernel: nodes [0, K) may live in shared memory for the duration
// of a launch (the fused kernel keeps the first, hottest nodes of every tree there: node indices grow
// in creation order, so the shallow levels every simulation walks through have the smallest indices);
// nodes >= K are in the HBM arena.  K == 0: everything in HBM.
// Shared-memory form of a node, 16 bytes = ONE load per child: value_sum, prior, and visit_count / first child as two
// 16-bit halves (so the lane that counts a visit and the lane that links the children store to different bytes).  Needs
// 1 + 7 * num_simulations <= 65535; larger searches run without the shared-memory prefix.
struct HotNode {
    double w;
    float p;
    uint16_t n, cb;
};
static_assert(sizeof(HotNode) == 16, "hot node record");

struct TreeMem {
    double *gW;
    uint4 *gM;
    HotNode *sH;
    uint32_t K;
#ifdef AZ_DEBUG_BOUNDS
    uint32_t cap;  // debug build (-DAZ_DEBUG_BOUNDS): every node access is checked against the tree's capacity
#endif
};
#ifdef AZ_DEBUG_BOUNDS
#define AZ_CHECK_NODE(tm, idx) assert((idx) < (tm).cap)
#define AZ_SET_CAP(tm, c) (tm).cap = (uint32_t)(c)
#else
#define AZ_CHECK_NODE(tm, idx) do { } while (0)
#define AZ_SET_CAP(tm, c) do { } while (0)
#endif

template <bool LAT>
__device__ __forceinline__ Child load_child(const TreeMem &tm, uint32_t idx, const Tabs &tb, double c_puct, double sq_parent) {
    Child ch;
    uint4 m;
    AZ_CHECK_NODE(tm, idx);
    if (idx < tm.K) {
        m = *reinterpret_cast<const uint4 *>(tm.sH + idx);
        ch.w = __hiloint2double((int)m.y, (int)m.x);
        ch.p = __uint_as_float(m.z);
        ch.n = m.w & 0xFFFFu;
        ch.cb = m.w >> 16;
    } else {
        m = tm.gM[idx];
        ch.w = tm.gW[idx];
        ch.n = m.x;
        ch.p = __uint_as_float(m.y);
        ch.cb = m.z;
    }
    // latency variant: everything the score needs from the tables is requested the moment the visit count is known, in one
    // round (the reciprocals used to be fetched inside the score, the second behind the first division's dependent chain)
    if (LAT) {
        const double2 e = tb.t2[ch.n];
        ch.r1 = e.x;
        ch.sq = e.y;
        ch.r0 = tb.rcp[ch.n];
        ch.x = __dmul_rn(__dmul_rn(c_puct, (double)ch.p), sq_parent);
        ch.d1 = (double)(1u + ch.n);
        ch.d0 = (double)ch.n;
    } else {
        ch.r1 = ch.r0 = ch.sq = ch.x = ch.d1 = ch.d0 = 0.0;
    }
    return ch;
}

__device__ __forceinline__ void store_new_child(const TreeMem &tm, uint32_t idx, float prior) {
    AZ_CHECK_NODE(tm, idx);
    const uint4 m = make_uint4(0u, __float_as_uint(prior), 0u, 0u);
    if (idx < tm.K) {
        *reinterpret_cast<uint4 *>(tm.sH + idx) = make_uint4(0u, 0u, __float_as_uint(prior), 0u);
    } else {
        tm.gW[idx] = 0.0;
        tm.gM[idx] = m;
    }
}

__device__ __forceinline__ void set_first_child(const TreeMem &tm, uint32_t idx, uint32_t first) {
    AZ_CHECK_NODE(tm, idx);
    if (idx < tm.K) tm.sH[idx].cb = (uint16_t)first;
    else reinterpret_cast<uint32_t *>(tm.gM + idx)[2] = first;
}

__device__ __forceinline__ void visit_node(const TreeMem &tm, uint32_t idx, double dv) {
    AZ_CHECK_NODE(tm, idx);
    if (idx < tm.K) {
        tm.sH[idx].w = __dadd_rn(tm.sH[idx].w, dv);
        tm.sH[idx].n += 1;
    } else {
        tm.gW[idx] = __dadd_rn(tm.gW[idx], dv);
        reinterpret_cast<uint32_t *>(tm.gM + idx)[0] += 1u;
    }
}

struct Leaf {
    uint64_t b0, b1;
    uint32_t node;
    int pl;     // side to move at the leaf
    int depth;  // number of moves below the root
    int first_col;  // column chosen at the root (valid when depth >= 1)
    bool win;   // the move into the leaf made 4-in-line (mover = pl ^ 1)
    bool term;  // win or board full
};

// AlphaZeroSearch.select_child repeated until an unexpanded node (search.py:72-73, 27-46).
// Warp-converged: every lane of the warp calls this; `alive` is uniform per quarter.  On entry
// (cb, sq_parent = sqrt(N)) describe the root and (root_legal, ch) hold the root's legal mask and this lane's
// root child record (valid when alive && cb != 0) — the fused kernel keeps them in registers across
// simulations.  `path[d]` receives the node index at depth d (written by lane 0 of the tree's lanes).
// LAT = true: the latency-optimised variant, for launches with few warps per SM (a simulation is one long dependent chain
// and nothing else hides it); LAT = false: fewer shuffles and loads per level, for launches that fill the issue slots.
// Measured on B200 (sims/s, 200 sims/move): 4096 trees 1.97e9 vs 1.81e9; 16384 trees 3.78e9 vs 4.45e9.
template <bool LAT>
__device__ __forceinline__ Leaf descend(const TreeMem &tm, const Tabs &tb,
                                        uint64_t rb0, uint64_t rb1, int rpl, double c_puct, uint32_t cb,
                                        double sq_parent, unsigned legal, Child ch, bool alive, bool writer,
                                        uint32_t *path, uint32_t &levels, uint32_t &scanned) {
    const int lane = threadIdx.x & 31;
    const int sub = lane & 24;
    const int c = lane & 7;
    const unsigned below = (1u << c) - 1u;
    Leaf L;
    L.b0 = rb0;
    L.b1 = rb1;
    L.pl = rpl;
    L.node = 0;
    L.depth = 0;
    L.first_col = 0;
    bool go = alive && cb != 0;
    bool my_legal = (legal >> c) & 1u;
    // The loop body is straight-line code: four trees share a warp and an idle eighth lane sits in every tree, so every
    // `if` here would be a divergent branch with its reconvergence barrier on the dependent chain.  Lanes of finished
    // trees keep computing on stale (valid) values and every update of the leaf is masked by `go`.
    // Dependent chain of one level: child record -> {rcp[n + 1], sqrt(n)}, rcp[n] -> PUCT (6 fp64 operations) -> 3 butterfly rounds ->
    // shuffle of the winner's first-child index -> next child record.  Everything else hangs off that chain: the
    // winner's sqrt comes with its record, the next node's legal mask is the current one minus the winning column if
    // that column fills up (known before the winner is), and the board update runs in the shadow of the next load.
    while (__any_sync(FULL, go)) {
        const uint64_t occ = L.b0 | L.b1;
        // columns with exactly five stones: one more and they leave the legal mask
        const bool fills = ((occ >> (c4::STRIDE * c + 4)) & 3ull) == 1ull;
        const unsigned fill_mask = (__ballot_sync(FULL, fills) >> sub) & 0x7Fu;
        const double s = LAT ? puct_score_pre(ch) : puct_score(ch.n, ch.w, ch.p, sq_parent, c_puct, tb.rcp);
        const double masked = (go && my_legal) ? s : -INFINITY;
        const int bc = LAT ? argmax_first(masked, c) : argmax_first_ballot(masked, sub);
        const uint32_t cb_sel = __shfl_sync(FULL, ch.cb, sub + bc);
        if (LAT) sq_parent = __shfl_sync(FULL, ch.sq, sub + bc);
        else sq_parent = tb.t2[__shfl_sync(FULL, ch.n, sub + bc)].y;
        const unsigned bcbit = 1u << bc;
        const unsigned lg = legal & ~(fill_mask & bcbit);  // legal mask of the node being entered
        const bool go_next = go && cb_sel != 0;
        const bool can = (lg >> c) & 1u;
        // The record to fetch: the winner's children start at cb_sel, this lane's is the popc-th of them.  Lanes that are not
        // legal there, or whose tree has finished, read node 0 (mask known before cb_sel arrives); if the winner turns out to
        // be unexpanded (cb_sel == 0) the lane reads node popc <= 6 of its own tree - the root or one of the root's children,
        // all initialised, since a descent only runs below an expanded root - and nothing of it is used (go_next is false).
        const uint32_t pre = (go && can) ? 0xFFFFFFFFu : 0u;
        const Child nxt = load_child<LAT>(tm, (cb_sel + (uint32_t)__popc(lg & below)) & pre, tb, c_puct, sq_parent);
        // Action.sample_next_state(): drop in column bc, flip the side to move
        const uint64_t bit = c4::drop_bit(occ, bc) & (0ull - (uint64_t)go);  // arithmetic mask: an `if (go)` here became a divergent branch
        const uint64_t bit0 = L.pl == 0 ? bit : 0ull;
        L.b0 |= bit0;
        L.b1 |= bit ^ bit0;
        L.pl ^= (int)go;
        const uint32_t entered = cb + __popc(legal & (bcbit - 1u));
        L.node = go ? entered : L.node;
        L.first_col = (go && L.depth == 0) ? bc : L.first_col;
        if (go && writer) path[L.depth + 1] = entered;
        L.depth += (int)go;
        levels += (uint32_t)go;
        scanned += go ? (uint32_t)__popc(legal) : 0u;
        cb = cb_sel;
        go = go_next;
        legal = lg;
        my_legal = can;
        ch = nxt;
    }
    // Node.is_terminal of the leaf (node.py:61-63).  Interior nodes are never terminal (a terminal
    // node is never expanded), so only the last mover's stones need the line test.
    // At depth 0 the leaf is the root itself, which has not ended (such trees are not alive): the test is false there as well,
    // so it runs unconditionally (an `if (depth > 0)` here is a branch with a reconvergence point on every simulation's chain).
    L.win = c4::has4_nb(L.pl ? L.b0 : L.b1);  // mover = pl ^ 1
    L.term = L.win || c4::is_full(L.b0 | L.b1);
    return L;
}

// AlphaZeroSearch.backpropagate (search.py:48-57) along the recorded path: the leaf gets +v, the sign
// flips going up except across a terminal leaf.  Stops at the current root (older ancestors are never
// read again, SURVEY App. A.5).  `lit` = lane index within the tree's lanes, `nl` = lanes per tree.
__device__ __forceinline__ void backup(const TreeMem &tm, const uint32_t *path, int depth, double v, bool leaf_terminal,
                                       int lit, int nl) {
    for (int i = lit; i <= depth; i += nl) {
        const int d = depth - i;
        const bool neg = leaf_terminal ? (d >= 1 && ((d - 1) & 1)) : (d & 1);
        visit_node(tm, path[i], neg ? -v : v);
    }
}

__device__ __forceinline__ double backup_sign(double v, int depth, int i, bool leaf_terminal) {
    const int d = depth - i;
    const bool neg = leaf_terminal ? (d >= 1 && ((d - 1) & 1)) : (d & 1);
    return neg ? -v : v;
}

// ------------------------------------------------------------------------------------------------
// fused search: all S simulations of a tree in one launch, built-in evaluator.
// The root's scalars (N, first child, legal mask) and each lane's root-child record live in registers
// for the whole launch, the first K nodes of every tree in shared memory (loaded at entry, written back
// at exit unless the launch also plays the move), the rest in HBM.  Dynamic shared memory: [TREES][K] HotNode (16 B),
// [TREES][44] u32 path, then (TSM) the tables: [tab_n] {1/(n+1), sqrt n} pairs (16 B), [tab_n] 1/d (8 B).
#ifdef AZ_TRUNK_CLOCKS
__device__ long long g_run_clk[8];
#define RCLK(var) const long long var = clock64()
#define RACC(i, t1, t0) do { racc[i] += (t1) - (t0); } while (0)
#else
#define RCLK(var) do { } while (0)
#define RACC(i, t1, t0) do { } while (0)
#endif

__device__ __forceinline__ void reset_tree(const Arena &a, int t) {
    const size_t base = (size_t)t * a.cap;
    a.W[base] = 0.0;
    a.M[base] = make_uint4(0u, 0u, 0u, 0u);
    a.used[t] = 1u;
}

// MOVE = true: the launch also plays the self-play move of every tree (what k_sample_moves does) - the root's child
// statistics are still in registers, the step's uniform and the game-log position were fetched at kernel entry, and the
// tree is discarded anyway (node.py:37-41), so the hot prefix is not written back.
__constant__ float c_inv_k[8] = {0.0f, 1.0f, 1.0f / 2.0f, 1.0f / 3.0f, 1.0f / 4.0f, 1.0f / 5.0f, 1.0f / 6.0f, 1.0f / 7.0f};

struct MoveArgs {
    const double *uniforms;
    uint8_t *finished;
    uint64_t init0, init1;
    int step, initpl;
};

// TSM: the tables live in shared memory (a compile-time fact, so that the loads are LDS, not generic loads)
// BUDGET (az_set_playout_cap; MOVE = false only): a tree takes part in a simulation only while its root has fewer visits than
// budget[t] (a trailing argument, so that the other builds keep their parameter layout); the other trees of the warp go on, and a
// warp whose trees have all reached their budget leaves the loop
template <int TPW, int EVAL, bool LAT, bool MOVE, bool TSM, bool BUDGET>
__global__ void __launch_bounds__(64) k_run_sims(Arena a, int n_active, int S, double c_puct, int K, MoveArgs mv, const uint32_t *budget) {
    constexpr int TREES = 2 * TPW;  // per 64-thread block
    constexpr int NL = 32 / TPW;    // lanes per tree
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int sub = lane & 24;
    const int c = lane & 7;
    const int q = lane / (32 / TPW);
    const int tib = warp * TPW + q;
    const int t = blockIdx.x * TREES + tib;
    // 1/d and sqrt(n) tables: every level's chain goes through them, and in L1 they compete with the node traffic (an L1 miss
    // costs an L2 round trip on the chain), so the block keeps its own copy in shared memory when they are small enough
    Tabs tb;
    if (TSM) {  // before any warp can leave: both warps of the block take part
        double2 *s_t2 = reinterpret_cast<double2 *>(smem_raw + (size_t)TREES * (K * sizeof(HotNode) + PATH_STRIDE * sizeof(uint32_t)));
        double *s_rcp = reinterpret_cast<double *>(s_t2 + a.tab_n);
        for (int i = threadIdx.x; i < a.tab_n; i += 64) {
            s_t2[i] = a.t2[i];
            s_rcp[i] = a.rcp[i];
        }
        tb.t2 = s_t2;
        tb.rcp = s_rcp;
        __syncthreads();
    } else {
        tb.t2 = a.t2;
        tb.rcp = a.rcp;
    }
    const bool alive = (t < n_active) && (a.tree_err[t < n_active ? t : 0] == 0);
    const int lit = lane & (NL - 1);
    if (MOVE && t < n_active && lit == 0 && mv.finished) mv.finished[t] = 0;
    if (!__any_sync(FULL, alive)) return;
    const int tt = alive ? t : 0;
    const bool writer = alive && lit == 0;
    const bool first_q = lit < 8;

    const size_t base = (size_t)tt * a.cap;
    TreeMem tm;
    tm.gW = a.W + base;
    tm.gM = a.M + base;
    tm.sH = reinterpret_cast<HotNode *>(smem_raw) + (size_t)tib * K;
    tm.K = (uint32_t)K;
    AZ_SET_CAP(tm, a.cap);
    uint32_t *path = reinterpret_cast<uint32_t *>(smem_raw + (size_t)TREES * K * sizeof(HotNode)) + tib * PATH_STRIDE;
    const uint64_t rb0 = a.root_bb0[tt], rb1 = a.root_bb1[tt];
    const int rpl = a.root_player[tt];
    uint32_t used = a.used[tt];
    uint32_t levels = 0, evals = 0, children = 0, scanned = 0;
    const uint32_t bud = BUDGET ? budget[tt] : 0u;
    double mv_u = 0.0;
    int mv_len = 0;
    if (MOVE && alive) {
        mv_u = mv.uniforms[t];
        mv_len = a.g_len[t];
    }

    // hot prefix of the tree -> shared memory.  Lanes without a tree of their own (tt = 0) fill their slot with tree 0's
    // records: the straight-line code below lets every lane load and score (masked), so what it reads must be valid.
    {
        const uint32_t hot = used < tm.K ? used : tm.K;
        for (uint32_t i = lit; i < hot; i += NL) {
            const uint4 m = tm.gM[i];
            HotNode hn;
            hn.w = tm.gW[i];
            hn.p = __uint_as_float(m.y);
            hn.n = (uint16_t)m.x;
            hn.cb = (uint16_t)m.z;
            tm.sH[i] = hn;
        }
        if (hot == 0 && lit == 0 && tm.K > 0) *reinterpret_cast<uint4 *>(tm.sH) = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncwarp();

    // root registers
    uint32_t root_n, root_cb;
    if (K > 0) {
        root_n = tm.sH[0].n;
        root_cb = tm.sH[0].cb;
    } else {
        const uint4 rm = tm.gM[0];
        root_n = rm.x;
        root_cb = rm.z;
    }
    const uint32_t n0 = root_n;  // BUDGET: every simulation adds one root visit, so the simulations run are root_n - n0 at the end
    const bool r_can = (c < c4::W) && !(((rb0 | rb1) >> (c4::STRIDE * c + 5)) & 1ull);
    const unsigned r_legal = (__ballot_sync(FULL, r_can) >> sub) & 0x7Fu;
    const int r_j = __popc(r_legal & ((1u << c) - 1u));
    Child rch;
    rch.w = 0.0; rch.sq = 0.0; rch.r1 = 1.0; rch.r0 = 0.0; rch.x = 0.0; rch.d1 = 1.0; rch.d0 = 0.0; rch.n = 0; rch.cb = 0; rch.p = 0.0f;
    double root_sq = tb.t2[root_n].y;
    if (alive && root_cb != 0 && r_can) rch = load_child<LAT>(tm, root_cb + r_j, tb, c_puct, root_sq);
    if (writer) path[0] = 0;

#ifdef AZ_TRUNK_CLOCKS
    long long racc[4] = {0, 0, 0, 0};
#endif
    for (int s = 0; s < S; ++s) {
        // the tree's part in this simulation: `live` stands for `alive` everywhere in the loop
        const bool live = BUDGET ? alive && root_n < bud : alive;
        if (BUDGET && !__any_sync(FULL, live)) break;
        RCLK(c0);
        Leaf L = descend<LAT>(tm, tb, rb0, rb1, rpl, c_puct, root_cb, root_sq, r_legal, rch, live, writer, path, levels, scanned);
        RCLK(c1);
        RACC(0, c1, c0);
        // Straight-line from here on as well (the four trees of a warp end in different cases).
        // Backup, part 1: lane `lit` owns path[lit]; its W / N loads are issued now and used after the expansion.  A leaf that
        // is expanded by this simulation is visited for the first time (N = 0, W = 0: a node is expanded on its first
        // visit), so it needs no load.
        __syncwarp();  // path[] (written by the tree's first lane) is visible to its other lanes
        const bool own = live && lit <= L.depth;
        const bool fresh = lit == L.depth && !L.term;
        const uint32_t my_idx = own ? path[lit] : 0u;
        const bool my_hot = my_idx < tm.K;
        double w_old = 0.0;
        uint32_t n_old = 0u;
        if (own && !fresh) {
            w_old = my_hot ? tm.sH[my_idx].w : tm.gW[my_idx];
            n_old = my_hot ? (uint32_t)tm.sH[my_idx].n : reinterpret_cast<const uint32_t *>(tm.gM + my_idx)[0];
        }
        // leaf: evaluate + expand, or terminal value
        const uint64_t occ = L.b0 | L.b1;
        const bool can = (c < c4::W) && !((occ >> (c4::STRIDE * c + 5)) & 1ull);
        const unsigned legal = (__ballot_sync(FULL, can) >> sub) & 0x7Fu;
        const int k = __popc(legal);
        const int j = __popc(legal & ((1u << c) - 1u));
        float prior, val;
        if (EVAL == AZ_EVAL_UNIFORM) {
            // fp32(1) / fp32(k), k = 1..7: compile-time constants from a constant-memory table (no MUFU slow path, no branches)
            prior = c_inv_k[k & 7];
            val = 0.0f;
        } else {
            const uint64_t h = azeval::board_hash(L.b0, L.b1, L.pl);
            prior = __fdiv_rn((float)azeval::hash_weight(h, c), (float)azeval::hash_weight_total(h, legal));
            const float v0 = azeval::hash_value0(h);
            val = L.pl == 0 ? v0 : -v0;
        }
        const bool expand = live && !L.term;
        if (expand && can && first_q) store_new_child(tm, used + j, prior);
        if (expand && writer) set_first_child(tm, L.node, used);
        // the root itself was expanded: its children enter the registers; depth 1: the chosen root child got children
        const bool root_exp = expand && L.depth == 0;
        const bool mine = L.depth >= 1 && c == L.first_col;
        root_cb = root_exp ? used : root_cb;
        rch.w = root_exp ? 0.0 : rch.w;
        rch.n = root_exp ? 0u : rch.n;  // (rch.sq follows rch.n below)
        rch.p = root_exp ? prior : rch.p;
        rch.cb = root_exp ? 0u : ((expand && mine && L.depth == 1) ? used : rch.cb);
        used += expand ? (uint32_t)k : 0u;
        children += expand ? (uint32_t)k : 0u;
        evals += (uint32_t)expand;
        // terminal leaf: reward[parent.state.player], the mover's own reward, +1 on a win, 0 on a draw (search.py:76);
        // otherwise value[node.state.player] (search.py:91)
        const double v = L.term ? (L.win ? 1.0 : 0.0) : (double)val;
        RCLK(c2);
        RACC(1, c2, c1);
        // Backup, part 2.  Registers: root and the chosen root child; memory: every node on the path.
        root_n += (uint32_t)live;
        root_sq = tb.t2[root_n].y;  // next simulation's sqrt(N_root) and the root child's table entries: loaded behind the backup
        rch.n += (uint32_t)(live && mine);
        if (LAT) {
            const double2 e = tb.t2[rch.n];
            rch.r1 = e.x;
            rch.sq = e.y;
            rch.r0 = tb.rcp[rch.n];
            rch.x = __dmul_rn(__dmul_rn(c_puct, (double)rch.p), root_sq);  // sqrt(N_root) changes with every simulation
            rch.d1 = (double)(1u + rch.n);
            rch.d0 = (double)rch.n;
        }
        rch.w = __dadd_rn(rch.w, (live && mine) ? backup_sign(v, L.depth, 1, L.term) : 0.0);  // + 0.0: value sums are never -0.0
        if (own) {
            const double w_new = __dadd_rn(w_old, backup_sign(v, L.depth, lit, L.term));
            if (my_hot) {
                tm.sH[my_idx].w = w_new;
                tm.sH[my_idx].n = (uint16_t)(n_old + 1u);
            } else {
                tm.gW[my_idx] = w_new;
                reinterpret_cast<uint32_t *>(tm.gM + my_idx)[0] = n_old + 1u;
            }
        }
        if (live)
            for (int i = lit + NL; i <= L.depth; i += NL) visit_node(tm, path[i], backup_sign(v, L.depth, i, L.term));
        __syncwarp();
        RCLK(c3);
        RACC(2, c3, c2);
        RACC(3, L.depth, 0);
    }
#ifdef AZ_TRUNK_CLOCKS
    if (blockIdx.x == 100 && threadIdx.x == 0)
        for (int i = 0; i < 4; ++i) g_run_clk[i] = racc[i];
#endif
    uint32_t moves = 0, episodes = 0;
    if (!MOVE) {
        // hot prefix back to the arena
        if (alive) {
            const uint32_t hot = used < tm.K ? used : tm.K;
            for (uint32_t i = lit; i < hot; i += NL) {
                const HotNode hn = tm.sH[i];
                tm.gM[i] = make_uint4(hn.n, __float_as_uint(hn.p), hn.cb, 0u);
                tm.gW[i] = hn.w;
            }
        }
    } else {
        // ---- the move step of this tree's game (episode_generator.py:53-78, node.py:23-42), same arithmetic as k_sample_moves
        RCLK(m0);
        const bool mover = alive && root_cb != 0;
        const int32_t cnt = (mover && r_can) ? (int32_t)rch.n : 0;
        const double p = __ddiv_rn((double)cnt, (double)((int)root_n - 1));  // improved_policy (node.py:27)
        double acc = 0.0, mycdf = 0.0;
        bool first = true;
#pragma unroll
        for (int j = 0; j < 7; ++j) {  // p.cumsum() over the legal columns, left to right
            const double pj = __shfl_sync(FULL, p, sub + j);
            const bool lj = (r_legal >> j) & 1u;
            acc = lj ? (first ? pj : __dadd_rn(acc, pj)) : acc;
            first = first && !lj;
            mycdf = (j == c) ? acc : mycdf;
        }
        // np.random.choice(k, p): cdf /= cdf[-1]; idx = searchsorted(cdf, u, side='right') = #{cdf <= u}
        const bool le = mover && r_can && __ddiv_rn(mycdf, acc) <= mv_u;
        int idx = __popc((__ballot_sync(FULL, le) >> sub) & 0x7Fu);
        const int k = __popc(r_legal);
        idx = idx >= k ? k - 1 : idx;
        const int col = c4::nth_legal_column(r_legal, idx < 0 ? 0 : idx);
        uint64_t nb0 = rb0, nb1 = rb1;
        const uint64_t bit = c4::drop_bit(rb0 | rb1, col);
        if (rpl == 0) nb0 |= bit; else nb1 |= bit;
        const bool win = c4::has4(rpl ? nb1 : nb0);
        const bool ended = win || c4::is_full(nb0 | nb1);
        const int new_len = mv_len + 1;
        // sample = (state, improved_policy) recorded before the move (episode_generator.py:56-62)
        if (mover && first_q && mv_len < MAX_PLIES) {
            const size_t o = (size_t)t * MAX_PLIES + mv_len;
            if (c < 7) a.g_counts[o * 7 + c] = cnt;
            if (lit == 0) {
                a.g_bb0[o] = rb0;
                a.g_bb1[o] = rb1;
                a.g_player[o] = (uint8_t)rpl;
            }
        }
        __syncwarp();
        RCLK(m1);
        long long dst = -1;
        if (mover && lit == 0) {
            moves = 1;
            if (!ended) {
                a.root_bb0[t] = nb0;
                a.root_bb1[t] = nb1;
                a.root_player[t] = (uint8_t)(rpl ^ 1);
                a.g_len[t] = new_len;
            } else {
                // outcome to every sample (episode.py:52-54); emit; recycle the slot (episode_generator.py:71-78)
                const int8_t r0 = win ? (rpl == 0 ? 1 : -1) : 0;
                const unsigned long long e = atomicAdd(&a.ring[0], 1ull);
                const unsigned long long o = atomicAdd(&a.ring[1], (unsigned long long)new_len);
                if ((long long)e < a.ep_cap && (long long)(o + new_len) <= a.s_cap) {
                    a.ep_slot[e] = t;
                    a.ep_step[e] = mv.step;
                    a.ep_len[e] = new_len;
                    a.ep_offset[e] = (int64_t)o;
                    a.ep_outcome[2 * e] = r0;
                    a.ep_outcome[2 * e + 1] = (int8_t)-r0;
                    dst = (long long)o;
                } else {
                    atomicAdd(&a.ring[2], 1ull);
                }
                episodes = 1;
                a.root_bb0[t] = mv.init0;
                a.root_bb1[t] = mv.init1;
                a.root_player[t] = (uint8_t)mv.initpl;
                a.g_len[t] = 0;
                if (mv.finished) mv.finished[t] = 1;
            }
            reset_tree(a, t);  // no subtree reuse: the new root has no children (node.py:37-41)
            used = 1u;
        }
        // the finished game's samples -> ring, one lane per sample
        RCLK(m2);
        dst = __shfl_sync(FULL, dst, lane - lit);
        if (dst >= 0) {
            const size_t g0 = (size_t)t * MAX_PLIES;
            for (int qq = lit; qq < new_len; qq += NL) {
                a.s_bb0[dst + qq] = a.g_bb0[g0 + qq];
                a.s_bb1[dst + qq] = a.g_bb1[g0 + qq];
                a.s_player[dst + qq] = a.g_player[g0 + qq];
#pragma unroll
                for (int i = 0; i < 7; ++i) a.s_counts[(dst + qq) * 7 + i] = a.g_counts[(g0 + qq) * 7 + i];
            }
        }
#ifdef AZ_TRUNK_CLOCKS
        {
            const long long m3 = clock64();
            if (blockIdx.x == 100 && threadIdx.x == 0) {
                g_run_clk[4] = m1 - m0; g_run_clk[5] = m2 - m1; g_run_clk[6] = m3 - m2;
            }
        }
#endif
    }
    if (writer) {
        a.used[t] = used;
        uint32_t *st = a.tstats + (size_t)t * NSTAT;
        st[0] += BUDGET ? root_n - n0 : (uint32_t)S;
        st[1] += evals;
        st[2] += levels;
        st[3] += children;
        st[4] += moves;
        st[5] += episodes;
        st[6] += scanned;
    }
}

// ------------------------------------------------------------------------------------------------
// evaluation cache (az_set_eval_cache).  The evaluator's row is a pure function of the position for a fixed set of weights, so a
// position evaluated before (same weights epoch) is served from the table, and a position that another tree claimed in the same
// selection launch reuses that tree's row: the search computes the same bits from fewer evaluator rows.
constexpr uint32_t CE_BUSY = 1, CE_PENDING = 2, CE_READY = 3;
constexpr uint32_t SRC_HIT = 0xFFFFFFFFu;   // leaf_src: the outputs are in cached_out
constexpr uint32_t NO_CLAIM = 0xFFFFFFFFu;  // leaf_claim: nothing to publish
constexpr uint32_t LAUNCH_MASK = 0x3FFFFFFFu;
constexpr int PROBE_ATTEMPTS = 8;  // re-reads of a bucket another tree is writing before the leaf is evaluated uncached

__device__ __forceinline__ unsigned long long ce_ctrl(uint32_t kind, uint32_t launch, uint32_t slot) {
    return (unsigned long long)kind | ((unsigned long long)(launch & LAUNCH_MASK) << 2) | ((unsigned long long)slot << 32);
}
__device__ __forceinline__ uint32_t ce_kind(unsigned long long c) { return (uint32_t)c & 3u; }
__device__ __forceinline__ uint32_t ce_launch(unsigned long long c) { return ((uint32_t)c >> 2) & LAUNCH_MASK; }

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint4 ld_volatile_v4(const void *p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long atom_add_acq_rel_u64(unsigned long long *p, unsigned long long v) {
    unsigned long long old;
    asm volatile("atom.acq_rel.gpu.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
    return old;
}

// The launch number and weights epoch of this launch, read by lane 0 of the warp (the lane whose ticket atomic in
// k_expand_select<COMPACT> orders the read before the last warp advances the launch number) and broadcast.
__device__ __forceinline__ void load_cache_ctl(const Arena &a, uint32_t &launch, uint32_t &epoch) {
    uint32_t l = 0, e = 0;
    if ((threadIdx.x & 31) == 0) {
        l = *reinterpret_cast<const volatile uint32_t *>(a.cache_ctl);
        e = *reinterpret_cast<const volatile uint32_t *>(a.cache_ctl + 1);
    }
    launch = __shfl_sync(FULL, l, 0);
    epoch = __shfl_sync(FULL, e, 0);
}

// Probe of slot t's non-terminal leaf (one lane per tree).  Returns the leaf's status: AZ_LEAF_SERVED for a hit (outputs copied to
// cached_out[t]) or a follower (leaf_src[t] = the slot whose row it reuses), AZ_LEAF_EVAL otherwise - with an entry claimed as
// PENDING for this launch (leaf_claim[t]; the expansion publishes the row there) unless every entry of the bucket is taken.
__device__ __forceinline__ uint8_t cache_probe(const Arena &a, int t, uint64_t b0, uint64_t b1, int pl, uint32_t launch, uint32_t epoch,
                                            uint32_t *st) {
    const uint32_t tag = epoch * 2u + (uint32_t)pl;
    const uint64_t h = azeval::mix64(b0 ^ azeval::mix64(b1 + (uint64_t)tag));
    CacheEntry *bk = a.cache + 2 * (size_t)((uint32_t)h & a.cache_mask);
    const uint32_t now = launch & LAUNCH_MASK;
    uint32_t claim = NO_CLAIM, src = (uint32_t)t;
    uint8_t status = AZ_LEAF_EVAL;
    int outcome = 2;  // st[] column - 7: 0 hit, 1 follower, 2 failed claim
    for (int attempt = 0; attempt < PROBE_ATTEMPTS; ++attempt) {
        if (attempt) __nanosleep(64);
        unsigned long long c[2];
        uint4 key[2], meta[2];  // {b0, b1}, {v1, tag, ctrl}
#pragma unroll
        for (int e = 0; e < 2; ++e) c[e] = ld_acquire_u64(&bk[e].ctrl);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            key[e] = ld_volatile_v4(&bk[e].b0);
            meta[e] = ld_volatile_v4(&bk[e].v1);
        }
        int match = -1, victim = -1;
        bool busy = false, evict = false;
        uint32_t best_age = 0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const uint32_t kind = ce_kind(c[e]);
            const bool same = key[e].x == (uint32_t)b0 && key[e].y == (uint32_t)(b0 >> 32) && key[e].z == (uint32_t)b1 &&
                              key[e].w == (uint32_t)(b1 >> 32) && meta[e].y == tag;
            const bool live_pending = kind == CE_PENDING && ce_launch(c[e]) == now;  // claimed in this launch: its row is coming
            if (same && (kind == CE_READY || live_pending) && match < 0) match = e;
            busy = busy || kind == CE_BUSY;
            if (kind == CE_BUSY || live_pending) continue;
            // free first (empty, a claim of an earlier launch, an older epoch's result), else the least recently published
            const bool current = kind == CE_READY && (meta[e].y >> 1) == epoch;
            const uint32_t age = current ? ((now - ce_launch(c[e])) & LAUNCH_MASK) : 0xFFFFFFFFu;
            if (victim < 0 || age > best_age) {
                victim = e;
                best_age = age;
                evict = current;
            }
        }
        if (match >= 0) {  // (selects, not indexing: the arrays stay in registers)
            const CacheEntry *m = bk + match;
            const unsigned long long cm = match ? c[1] : c[0];
            uint4 p0 = make_uint4(0u, 0u, 0u, 0u), p1 = p0;
            const bool hit = ce_kind(cm) == CE_READY;
            if (hit) {
                p0 = ld_volatile_v4(&m->p0);
                p1 = ld_volatile_v4(&m->p1);
            }
            __threadfence();
            if (ld_relaxed_u64(&m->ctrl) != cm) continue;  // rewritten while we read it
            if (hit) {
                a.cached_out[(size_t)t * 3] = make_float4(__uint_as_float(p0.x), __uint_as_float(p0.y), __uint_as_float(p0.z), __uint_as_float(p0.w));
                a.cached_out[(size_t)t * 3 + 1] = make_float4(__uint_as_float(p1.x), __uint_as_float(p1.y), __uint_as_float(p1.z), __uint_as_float(p1.w));
                a.cached_out[(size_t)t * 3 + 2] = make_float4(__uint_as_float(match ? meta[1].x : meta[0].x), 0.0f, 0.0f, 0.0f);
                src = SRC_HIT;
                outcome = 0;
            } else {
                src = (uint32_t)(cm >> 32);
                outcome = 1;
            }
            status = AZ_LEAF_SERVED;
            break;
        }
        if (busy || victim < 0) continue;  // another tree is writing this bucket (perhaps this position): look again
        CacheEntry *v = bk + victim;
        const unsigned long long cv = victim ? c[1] : c[0];
        if (atomicCAS(&v->ctrl, cv, ce_ctrl(CE_BUSY, now, (uint32_t)t)) != cv) continue;
        __threadfence();
        v->b0 = b0;
        v->b1 = b1;
        v->tag = tag;
        __threadfence();
        *reinterpret_cast<volatile unsigned long long *>(&v->ctrl) = ce_ctrl(CE_PENDING, now, (uint32_t)t);
        claim = (uint32_t)(v - a.cache);
        st[10] += evict ? 1u : 0u;
        outcome = -1;
        break;
    }
    if (outcome >= 0) st[7 + outcome] += 1u;
    a.leaf_src[t] = src;
    a.leaf_claim[t] = claim;
    return status;
}

// The expansion of a leaf that claimed entry `claim` in the previous launch publishes its row there (one lane per tree); a claim
// that another tree has taken over meanwhile (it counts as empty one launch later) is dropped.
__device__ __forceinline__ void cache_publish(const Arena &a, uint32_t claim, int t, uint32_t launch, float4 p0, float4 p1, float v1) {
    CacheEntry *e = a.cache + claim;
    const unsigned long long want = ce_ctrl(CE_PENDING, launch - 1u, (uint32_t)t);
    if (atomicCAS(&e->ctrl, want, ce_ctrl(CE_BUSY, launch, (uint32_t)t)) != want) return;
    __threadfence();
    e->p0 = p0;
    e->p1 = p1;
    e->v1 = v1;
    __threadfence();
    *reinterpret_cast<volatile unsigned long long *>(&e->ctrl) = ce_ctrl(CE_READY, launch, (uint32_t)t);
}

// ------------------------------------------------------------------------------------------------
// split path, step 1: search.py:69-79
// CACHE: non-terminal leaves are probed in the evaluation cache; launch / epoch from load_cache_ctl
// SYM: a non-terminal leaf is written (and probed) in its canonical form, leaf_mirror[t] = 1 when that is its mirror (the array
// is a trailing kernel argument rather than an Arena member, so that the other kernels' parameter layout stays as it was); every
// evaluator then evaluates the canonical position, so the search runs with f_sym(x) = unmirror_if_flagged(f(canon(x)))
// BUDGET (az_set_playout_cap): a tree whose root has reached its visit budget (budget[t], a trailing kernel argument like
// leaf_mirror) has finished its search of this move step and is idle, as a tree in error is: every simulation adds exactly one
// visit to the root, so the root's N counts the simulations done
template <int TPW, bool LAT, bool CACHE, bool SYM, bool BUDGET>
__device__ __forceinline__ bool select_body(const Arena &a, int n_active, double c_puct, uint32_t launch, uint32_t epoch,
                                            uint8_t *leaf_mirror, const uint32_t *budget) {
    constexpr int TREES = 2 * TPW;
    constexpr int NL = 32 / TPW;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int sub = lane & 24;
    const int c = lane & 7;
    const int q = lane / (32 / TPW);
    const int t = blockIdx.x * TREES + warp * TPW + q;
    const bool in_range = t < n_active;
    const int tt = in_range ? t : 0;
    const size_t base = (size_t)tt * a.cap;
    TreeMem tm;
    tm.gW = a.W + base;
    tm.gM = a.M + base;
    tm.sH = nullptr;
    tm.K = 0;
    AZ_SET_CAP(tm, a.cap);
    // first round of loads, all independent: error flag, root position, root record (and the visit budget)
    const int32_t err = a.tree_err[tt];
    const uint64_t rb0 = a.root_bb0[tt], rb1 = a.root_bb1[tt];
    const int rpl = a.root_player[tt];
    const uint4 rm = tm.gM[0];
    const uint32_t bud = BUDGET ? budget[tt] : 0u;
    const bool alive = in_range && err == 0 && (!BUDGET || rm.x < bud);
    const int lit = lane & (NL - 1);
    if (in_range && !alive && lit == 0) {
        a.leaf_status[t] = AZ_LEAF_IDLE;
        if (SYM) leaf_mirror[t] = 0;
    }
    if (!__any_sync(FULL, alive)) return false;
    const bool writer = alive && lit == 0;
    uint32_t *path = a.path + (size_t)tt * PATH_STRIDE;
    const bool r_can = (c < c4::W) && !(((rb0 | rb1) >> (c4::STRIDE * c + 5)) & 1ull);
    const unsigned r_legal = (__ballot_sync(FULL, r_can) >> sub) & 0x7Fu;
    Child rch;
    rch.w = 0.0; rch.sq = 0.0; rch.r1 = 1.0; rch.r0 = 0.0; rch.x = 0.0; rch.d1 = 1.0; rch.d0 = 0.0; rch.n = 0; rch.cb = 0; rch.p = 0.0f;
    Tabs tb;
    tb.rcp = a.rcp;
    tb.t2 = a.t2;
    const double root_sq = __ldg(a.sqt + rm.x);
    if (alive && rm.z != 0 && r_can) rch = load_child<LAT>(tm, rm.z + __popc(r_legal & ((1u << c) - 1u)), tb, c_puct, root_sq);
    if (writer) path[0] = 0;
    uint32_t levels = 0, scanned = 0;
    Leaf L = descend<LAT>(tm, tb, rb0, rb1, rpl, c_puct, rm.z, root_sq, r_legal, rch, alive, writer, path, levels, scanned);
    uint8_t status = L.term ? AZ_LEAF_TERMINAL : AZ_LEAF_EVAL;
    if (writer) {
        uint32_t *st = a.tstats + (size_t)t * NSTAT;
        uint64_t lb0 = L.b0, lb1 = L.b1;
        if (SYM) {
            const c4::Canonical k = c4::canonical(L.b0, L.b1);
            const bool mir = k.mirrored && !L.term;
            lb0 = mir ? k.b0 : L.b0;
            lb1 = mir ? k.b1 : L.b1;
            leaf_mirror[t] = mir ? 1 : 0;
        }
        if (CACHE && !L.term) status = cache_probe(a, t, lb0, lb1, L.pl, launch, epoch, st);
        a.leaf_node[t] = L.node;
        a.leaf_bb0[t] = lb0;
        a.leaf_bb1[t] = lb1;
        a.leaf_player[t] = (uint8_t)L.pl;
        a.leaf_depth[t] = (uint8_t)L.depth;
        a.leaf_status[t] = status;
        st[0] += 1u;
        st[2] += levels;
        st[6] += scanned;
    }
    __syncwarp();
    if (alive && L.term) backup(tm, path, L.depth, L.win ? 1.0 : 0.0, true, lit, NL);
    return writer && status == AZ_LEAF_EVAL;  // this lane wrote AZ_LEAF_EVAL for its tree
}

// split path, step 3: search.py:87-91 with the evaluator's outputs
template <int TPW, bool LAT, bool CACHE, bool SYM, bool BUDGET>
__global__ void __launch_bounds__(64) k_select(Arena a, int n_active, double c_puct, uint8_t *leaf_mirror, const uint32_t *budget) {
    uint32_t launch = 0, epoch = 0;
    if (CACHE) load_cache_ctl(a, launch, epoch);
    select_body<TPW, LAT, CACHE, SYM, BUDGET>(a, n_active, c_puct, launch, epoch, leaf_mirror, budget);
}

// split path, step 3: search.py:87-91 with the evaluator's outputs
// CACHE: a SERVED leaf takes its outputs from cached_out or from its leader's row, and a leaf that claimed an entry publishes its row
// SYM: lane c works on column c of the canonical leaf the evaluator saw (legal mask, logit, softmax, published row); for a mirrored
// leaf that is actual column 6 - c, whose index among the actual children (ascending columns) is k - 1 - j instead of j
template <int TPW, bool CACHE, bool SYM>
__device__ __forceinline__ void expand_backup_body(const Arena &a, int n_active, const float *__restrict__ policy,
                                                   const float *__restrict__ values, int policy_kind, uint32_t launch,
                                                   const uint8_t *leaf_mirror) {
    constexpr int TREES = 2 * TPW;
    constexpr int NL = 32 / TPW;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int sub = lane & 24;
    const int c = lane & 7;
    const int q = lane / (32 / TPW);
    const int t = blockIdx.x * TREES + warp * TPW + q;
    // Every load that does not depend on another is issued in the first round (the slot's leaf record, the evaluator's
    // outputs, this lane's path entry): the kernel is a chain of dependent HBM / L2 round trips, nothing else.
    const int tt = t < n_active ? t : 0;
    const int lit = lane & (NL - 1);
    const uint8_t status = a.leaf_status[tt];
    const uint64_t occ = a.leaf_bb0[tt] | a.leaf_bb1[tt];
    const int pl = a.leaf_player[tt];
    const uint32_t node = a.leaf_node[tt];
    const int depth = a.leaf_depth[tt];
    const uint32_t used = a.used[tt];
    const uint32_t *path = a.path + (size_t)tt * PATH_STRIDE;
    const uint32_t my_idx = path[lit < PATH_STRIDE ? lit : 0];
    float x_raw = policy[(size_t)tt * 7 + (c < 7 ? c : 0)];
    float v0 = values[(size_t)tt * 2], v1 = values[(size_t)tt * 2 + 1];
    const uint32_t src = CACHE ? a.leaf_src[tt] : 0u;
    const uint32_t claim = CACHE ? a.leaf_claim[tt] : NO_CLAIM;
    const bool mir = SYM && leaf_mirror[tt] != 0;
    const bool served = CACHE && status == AZ_LEAF_SERVED;
    const bool alive = (t < n_active) && (status == AZ_LEAF_EVAL || served);
    if (!__any_sync(FULL, alive)) return;
    if (served && alive) {  // the rows of SERVED leaves were not evaluated: the outputs are the leader's row or the cached copy
        const float *o = src == SRC_HIT ? reinterpret_cast<const float *>(a.cached_out + (size_t)tt * 3) : policy + (size_t)src * 7;
        x_raw = o[c < 7 ? c : 0];
        v0 = src == SRC_HIT ? o[7] : values[(size_t)src * 2];
        v1 = src == SRC_HIT ? o[8] : values[(size_t)src * 2 + 1];
    }
    const bool writer = alive && lit == 0;
    const bool first_q = lit < 8;
    const size_t base = (size_t)tt * a.cap;
    TreeMem tm;
    tm.gW = a.W + base;
    tm.gM = a.M + base;
    tm.sH = nullptr;
    tm.K = 0;
    AZ_SET_CAP(tm, a.cap);
    // second round: W / N of this lane's path node (the leaf itself is visited for the first time: nothing to load)
    const bool own = alive && lit <= depth;
    const bool fresh = lit == depth;
    double w_old = 0.0;
    uint32_t n_old = 0u;
    if (own && !fresh) {
        w_old = tm.gW[my_idx];
        n_old = reinterpret_cast<const uint32_t *>(tm.gM + my_idx)[0];
    }
    const bool can = (c < c4::W) && !((occ >> (c4::STRIDE * c + 5)) & 1ull);
    const unsigned legal = (__ballot_sync(FULL, can) >> sub) & 0x7Fu;
    const int k = __popc(legal);
    const int j = __popc(legal & ((1u << c) - 1u));
    const float x = (alive && can) ? x_raw : -INFINITY;
    float prior;
    if (policy_kind == AZ_POLICY_PRIORS) {
        prior = x;
    } else {
        // F.softmax over the logits of the legal columns only, fp32 (model.py:29-35)
        float m = x;
#pragma unroll
        for (int off = 4; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, off));
        const float e = (alive && can) ? expf(x - m) : 0.0f;
        float sum = e;
#pragma unroll
        for (int off = 4; off >= 1; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
        prior = __fdiv_rn(e, sum);
    }
    __syncwarp();  // every lane has read used / leaf_* before the writer updates them
    if (alive) {
        if (can && first_q) store_new_child(tm, used + (mir ? k - 1 - j : j), prior);
        const double v = (double)(pl ? v1 : v0);  // value[node.state.player] (search.py:91)
        if (writer) {
            set_first_child(tm, node, used);
            a.used[t] = used + k;
            a.leaf_status[t] = AZ_LEAF_IDLE;  // consumed: a second az_expand_backup without a select is a no-op
            uint32_t *st = a.tstats + (size_t)t * NSTAT;
            st[1] += 1u;
            st[3] += (uint32_t)k;
        }
        if (own) {
            tm.gW[my_idx] = __dadd_rn(w_old, backup_sign(v, depth, lit, false));
            reinterpret_cast<uint32_t *>(tm.gM + my_idx)[0] = n_old + 1u;
        }
        for (int i = lit + NL; i <= depth; i += NL) visit_node(tm, path[i], backup_sign(v, depth, i, false));
    }
    if (CACHE) {
        const bool publish = alive && status == AZ_LEAF_EVAL && claim != NO_CLAIM;
        if (__any_sync(FULL, publish)) {
            const int l0 = lane - lit;  // the tree's first lane: lanes l0 + 0..6 hold the row's 7 logits
            float o[7];
#pragma unroll
            for (int j = 0; j < 7; ++j) o[j] = __shfl_sync(FULL, x_raw, l0 + j);
            if (publish && writer) cache_publish(a, claim, t, launch, make_float4(o[0], o[1], o[2], o[3]), make_float4(o[4], o[5], o[6], v0), v1);
        }
    }
}

template <int TPW, bool CACHE, bool SYM>
__global__ void __launch_bounds__(64)
k_expand_backup(Arena a, int n_active, const float *__restrict__ policy, const float *__restrict__ values, int policy_kind,
                const uint8_t *leaf_mirror) {
    uint32_t launch = 0, epoch = 0;
    if (CACHE) load_cache_ctl(a, launch, epoch);
    expand_backup_body<TPW, CACHE, SYM>(a, n_active, policy, values, policy_kind, launch, leaf_mirror);
}

// Steps 3 and 1 of consecutive simulations in one launch: expansion + backup of simulation k, then the selection of simulation
// k + 1 (same thread -> tree mapping in both, so a tree is only ever touched by its own warp; __syncwarp orders the two halves).
// One launch less per simulation step of the network-in-the-loop path.
// COMPACT: the list of the slots whose new leaf waits for the evaluator (what k_compact_leaves writes in one more launch) is built
// here.  One 64-bit atomic per warp on the word at eval_count[2..3]: the low half hands out list positions for the warp's up-to-TPW
// slots, the high half counts the warps that are through - the warp that finds every other warp's ticket taken publishes the total
// in eval_count[0] and zeroes the word for the next launch.  No fences: the next kernel on the stream is the first reader.  The
// list is a permutation of k_compact_leaves' ascending one (the order is the order of the tickets); the evaluators scatter their
// outputs to the slots' rows and a position's outputs do not depend on the batch it falls into, so the search is unchanged.
// CACHE: both halves use the evaluation cache; with COMPACT the last warp also advances the launch number (the ticket atomic is then
// acq_rel, so that every warp's read of the number at its start precedes the advance).
template <int TPW, bool LAT, bool COMPACT, bool CACHE, bool SYM, bool BUDGET>
__global__ void __launch_bounds__(64)
k_expand_select(Arena a, int n_active, const float *__restrict__ policy, const float *__restrict__ values, int policy_kind, double c_puct,
                uint8_t *leaf_mirror, const uint32_t *budget) {
    uint32_t launch = 0, epoch = 0;
    if (CACHE) load_cache_ctl(a, launch, epoch);
    expand_backup_body<TPW, CACHE, SYM>(a, n_active, policy, values, policy_kind, launch, leaf_mirror);
    __syncwarp();
    const bool wants = select_body<TPW, LAT, CACHE, SYM, BUDGET>(a, n_active, c_puct, launch, epoch, leaf_mirror, budget);
    if (COMPACT) {
        const int lane = threadIdx.x & 31;
        const unsigned m = __ballot_sync(FULL, wants);
        unsigned long long *word = reinterpret_cast<unsigned long long *>(a.eval_count + 2);
        unsigned long long old = 0ull;
        if (lane == 0) {
            const unsigned long long ticket = (1ull << 32) | (unsigned long long)__popc(m);
            old = CACHE ? atom_add_acq_rel_u64(word, ticket) : atomicAdd(word, ticket);
            if ((unsigned)(old >> 32) == gridDim.x * 2u - 1u) {  // every other warp of the launch has its ticket
                a.eval_count[0] = (int32_t)((unsigned)old + (unsigned)__popc(m));
                *word = 0ull;
                if (CACHE) a.cache_ctl[0] = launch + 1u;
            }
        }
        const int at = (int)__shfl_sync(FULL, (unsigned)old, 0);
        if (wants) a.eval_list[at + __popc(m & ((1u << lane) - 1u))] = blockIdx.x * (2 * TPW) + (threadIdx.x >> 5) * TPW + lane / (32 / TPW);
    }
}

// Ordered compaction of the slots whose leaf waits for the evaluator (status AZ_LEAF_EVAL): eval_list[0 .. count) ascending.
// ~15 % of the simulations of a running self-play loop end in a terminal leaf (search.py:75-77) and need no evaluation; the
// tensor-core evaluators walk this list instead of all E rows and scatter their outputs back to the slots' rows.  One block:
// each thread counts its contiguous stretch of slots, a block-wide exclusive scan gives its offset (deterministic order, no atomics).
// Thread t owns the slots [t * per, t * per + per), per a multiple of 16, and reads them as 16-byte vectors (the status array is
// padded by 16 bytes): one L2 round trip per thread instead of one per slot.
__device__ __forceinline__ uint32_t eval_bits(uint32_t w) { return ~(w | (w >> 1)) & 0x01010101u; }  // bit 8 i set <=> byte i == AZ_LEAF_EVAL (0); bytes are 0 .. 3
// `advance` (the evaluation cache's launch number, or null): one more selection launch is over.
__global__ void __launch_bounds__(1024) k_compact_leaves(const uint8_t *__restrict__ status, int n, int32_t *__restrict__ list, int32_t *__restrict__ count, int staged,
                                                         uint32_t *advance) {
    static_assert(AZ_LEAF_EVAL == 0 && AZ_LEAF_TERMINAL == 1 && AZ_LEAF_IDLE == 2 && AZ_LEAF_SERVED == 3, "eval_bits relies on the status encoding");
    __shared__ int warp_tot[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (advance && tid == 0) *advance += 1u;
    const int per = (((n + 1023) / 1024) + 15) & ~15;
    const int lo = tid * per;
    int mine = 0;
    for (int base = lo; base < lo + per && base < n; base += 16) {
        const uint4 v = *reinterpret_cast<const uint4 *>(status + base);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t z = eval_bits(w[k]);
            const int left = n - (base + 4 * k);  // slots of this word that exist
            if (left < 4) z &= left <= 0 ? 0u : (0x01010101u >> (8 * (4 - left)));
            mine += __popc(z);
        }
    }
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(FULL, incl, off);
        if (lane >= off) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = warp_tot[lane], wi = w;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_up_sync(FULL, wi, off);
            if (lane >= off) wi += v;
        }
        warp_tot[lane] = wi - w;  // exclusive
        if (lane == 31) count[0] = wi;
    }
    __syncthreads();
    if (per == 16 && staged) {
        // n <= 16384 (configs[2], configs[3] at 4 / 8 GPUs): a warp's 512 slots give one contiguous stretch of the list.  The entries
        // are staged in shared memory (as 16-bit offsets from the warp's first slot) and written with coalesced stores: one thread's
        // up-to-16 scattered 4-byte stores cost the SM ~30 sectors per store instruction - 12.2 -> 7.0 us per launch under ncu
        // (AZ_COMPACT_STAGE=0: the direct stores).
        __shared__ uint16_t stage[32][512];
        int o = incl - mine;  // offset inside the warp's stretch
        if (lo < n) {
            const uint4 v = *reinterpret_cast<const uint4 *>(status + lo);  // L1 hit
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t z = eval_bits(w[k]);
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int i = lo + 4 * k + b;
                    if (((z >> (8 * b)) & 1u) && i < n) stage[warp][o++] = (uint16_t)(16 * lane + 4 * k + b);
                }
            }
        }
        const int cnt = __shfl_sync(FULL, incl, 31);
        __syncwarp();
        const int out0 = warp_tot[warp], slot0 = warp * 512;
        for (int j = lane; j < cnt; j += 32) list[out0 + j] = slot0 + (int)stage[warp][j];
        return;
    }
    int o = warp_tot[warp] + incl - mine;
    for (int base = lo; base < lo + per && base < n; base += 16) {
        const uint4 v = *reinterpret_cast<const uint4 *>(status + base);  // L1 hit
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t z = eval_bits(w[k]);
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int i = base + 4 * k + b;
                if (((z >> (8 * b)) & 1u) && i < n) list[o++] = i;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// plane encoders (the "leaf gather").  One thread per position builds the position's output words from
// row-major plane masks (a handful of integer ops per word), stages them in shared memory, and the block
// then streams the staged tile to HBM with coalesced 16-byte stores: a tile of B positions is contiguous in
// the output, so the write side runs at copy speed regardless of the 252 / 168 / 504 / 672-byte record size.
__host__ __device__ inline int layout_elems(int layout) {
    return layout == AZ_LAYOUT_GRID_F32 ? 42 : (layout == AZ_LAYOUT_PLANES_BF16_NHWC ? 336 : 126);
}
__host__ __device__ inline int layout_words(int layout) {  // 32-bit words per position
    return layout == AZ_LAYOUT_GRID_F32 ? 42 : (layout == AZ_LAYOUT_PLANES_F32 ? 126 : (layout == AZ_LAYOUT_PLANES_BF16 ? 63 : 168));
}

// column-major bitboard (bit = 7*col + row) -> row-major 42-bit mask (bit = 7*row + col), the element order of [6][7]
__device__ __forceinline__ uint64_t to_row_major(uint64_t bb) {
    uint64_t m = 0;
#pragma unroll
    for (int r = 0; r < c4::H; ++r) {
        const uint64_t row = ((((bb >> r) & 0x40810204081ull) * c4::LEGAL_MAGIC) >> 36) & 0x7Full;
        m |= row << (7 * r);
    }
    return m;
}

template <int LAYOUT>
__global__ void __launch_bounds__(128)
k_encode(const uint64_t *__restrict__ bb0, const uint64_t *__restrict__ bb1, const uint8_t *__restrict__ player,
         const uint8_t *__restrict__ status, long long n, uint32_t *__restrict__ out) {
    constexpr int W = (LAYOUT == AZ_LAYOUT_GRID_F32) ? 42 : (LAYOUT == AZ_LAYOUT_PLANES_F32) ? 126 : (LAYOUT == AZ_LAYOUT_PLANES_BF16) ? 63 : 168;
    constexpr int WP = (W % 2 == 0) ? W + 1 : W;  // odd row stride: conflict-free staging
    extern __shared__ uint32_t s_tile[];          // [blockDim.x][WP]
    const int B = blockDim.x;
    const long long t0 = (long long)blockIdx.x * B;
    const long long t = t0 + threadIdx.x;
    uint32_t *row = s_tile + threadIdx.x * WP;
    if (t < n) {
        uint64_t b0 = bb0[t], b1 = bb1[t];
        const int pl = player[t] & 1;
        const bool live = status ? (status[t] == AZ_LEAF_EVAL || status[t] == AZ_LEAF_SERVED) : true;
        if (LAYOUT == AZ_LAYOUT_GRID_F32) {
            // state.grid as f32: -1 empty / 0 / 1 owner (basic.py:41-47)
            const uint64_t m0 = to_row_major(b0), m1 = to_row_major(b1);
#pragma unroll
            for (int e = 0; e < 42; ++e) {
                const uint32_t v = ((m0 >> e) & 1ull) ? 0x00000000u : (((m1 >> e) & 1ull) ? 0x3F800000u : 0xBF800000u);
                row[e] = live ? v : 0u;
            }
        } else {
            // planes: empty, side to move, opponent (cnn.py:93-95)
            const uint64_t mine = pl ? b1 : b0, theirs = pl ? b0 : b1;
            uint64_t p0 = to_row_major(~(b0 | b1) & c4::BOARD), p1 = to_row_major(mine), p2 = to_row_major(theirs);
            if (!live) p0 = p1 = p2 = 0;
            if (LAYOUT == AZ_LAYOUT_PLANES_F32) {
#pragma unroll
                for (int e = 0; e < 42; ++e) {
                    row[e] = ((p0 >> e) & 1ull) ? 0x3F800000u : 0u;
                    row[42 + e] = ((p1 >> e) & 1ull) ? 0x3F800000u : 0u;
                    row[84 + e] = ((p2 >> e) & 1ull) ? 0x3F800000u : 0u;
                }
            } else if (LAYOUT == AZ_LAYOUT_PLANES_BF16) {
                // 126 bf16 = 63 words; element stream = p0 (42 bits) | p1 (42) | p2 (42)
                const uint64_t lo = p0 | (p1 << 42);          // elements 0..63
                const uint64_t hi = (p1 >> 22) | (p2 << 20);  // elements 64..125
#pragma unroll
                for (int w = 0; w < 63; ++w) {
                    const uint32_t two = (w < 32) ? (uint32_t)(lo >> (2 * w)) & 3u : (uint32_t)(hi >> (2 * (w - 32))) & 3u;
                    row[w] = ((two & 1u) ? 0x00003F80u : 0u) | ((two & 2u) ? 0x3F800000u : 0u);
                }
            } else {  // NHWC, 8 channels per cell: c0 c1 | c2 0 | 0 0 | 0 0
#pragma unroll
                for (int e = 0; e < 42; ++e) {
                    row[4 * e] = (((p0 >> e) & 1ull) ? 0x00003F80u : 0u) | (((p1 >> e) & 1ull) ? 0x3F800000u : 0u);
                    row[4 * e + 1] = ((p2 >> e) & 1ull) ? 0x00003F80u : 0u;
                    row[4 * e + 2] = 0u;
                    row[4 * e + 3] = 0u;
                }
            }
        }
    }
    __syncthreads();
    const long long remaining = n - t0;
    const int valid = remaining < B ? (int)remaining : B;
    const int total_words = valid * W;
    uint32_t *dst = out + t0 * W;  // B*W*4 bytes per full tile: 16-byte aligned whenever B is a multiple of 4
    const int quads = total_words >> 2;
    for (int qd = threadIdx.x; qd < quads; qd += B) {
        uint32_t v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int w = 4 * qd + k;
            v[k] = s_tile[(w / W) * WP + (w % W)];
        }
        reinterpret_cast<uint4 *>(dst)[qd] = make_uint4(v[0], v[1], v[2], v[3]);
    }
    for (int w = 4 * quads + threadIdx.x; w < total_words; w += B) dst[w] = s_tile[(w / W) * WP + (w % W)];
}

// ------------------------------------------------------------------------------------------------
// rules kernels (one thread per position)
__global__ void __launch_bounds__(256)
k_env_step(const uint64_t *__restrict__ bb0, const uint64_t *__restrict__ bb1, const uint8_t *__restrict__ player,
           const uint8_t *__restrict__ col, long long n, uint64_t *o0, uint64_t *o1, uint8_t *opl, uint8_t *olegal,
           uint8_t *oended, int8_t *oreward, uint8_t *ostatus) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t b0 = bb0[i], b1 = bb1[i];
    int pl = player[i] & 1;
    const int cc = col[i];
    c4::Terminal T = c4::terminal_of(b0, b1);
    uint8_t status = 1;
    if (!T.ended && cc < c4::W && !(((b0 | b1) >> (c4::STRIDE * cc + 5)) & 1ull)) {
        const uint64_t bit = c4::drop_bit(b0 | b1, cc);
        if (pl == 0) b0 |= bit; else b1 |= bit;
        const bool win = c4::has4(pl ? b1 : b0);
        T.ended = win || c4::is_full(b0 | b1);
        T.reward0 = win ? (pl == 0 ? 1 : -1) : 0;
        pl ^= 1;
        status = 0;
    }
    if (o0) o0[i] = b0;
    if (o1) o1[i] = b1;
    if (opl) opl[i] = (uint8_t)pl;
    if (olegal) olegal[i] = T.ended ? 0 : (uint8_t)c4::legal_mask(b0 | b1);
    if (oended) oended[i] = T.ended ? 1 : 0;
    if (oreward) {
        oreward[2 * i] = T.reward0;
        oreward[2 * i + 1] = (int8_t)-T.reward0;
    }
    if (ostatus) ostatus[i] = status;
}

// 4 positions per thread: 128-bit loads / stores of the bitboards, 32-bit loads / stores of the byte arrays; used when every
// pointer is present and 16-byte aligned (the normal case), the scalar kernels cover the rest.  The rules run on the 32-bit halves
// of the boards (c4::h32): the 64-bit formulation compiles to ALU-pipe instructions only (697 per 4 positions in the first version
// of the step kernel) and that pipe bounded the kernels at 59 % / 53 % of HBM; with the low-word shifts, three directions' high-word
// shifts, the byte packing and the column arithmetic on the FMA pipe it is 424 ALU + 280 FMA (76 % / 76 %, profiles/r02_rules_kernels.json).
template <int MODE>
__global__ void __launch_bounds__(256)
k_env_step_h(const uint4 *__restrict__ bb0, const uint4 *__restrict__ bb1, const uint32_t *__restrict__ player,
             const uint32_t *__restrict__ col, long long quads, uint4 *o0, uint4 *o1, uint32_t *opl, uint32_t *olegal,
             uint32_t *oended, uint2 *oreward, uint32_t *ostatus) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= quads) return;
    const uint4 a0 = bb0[2 * i], a1 = bb0[2 * i + 1], c0 = bb1[2 * i], c1 = bb1[2 * i + 1];
    const uint32_t pw = player[i] & 0x01010101u, cw = col[i];
    using namespace c4::h32;
    const uint32_t px = mad_u32(pw, 0x80u, 0u);
    const Step s0 = env_step<MODE>(a0.x, a0.y, c0.x, c0.y, player_mask(px, 0), byte_of(cw, 0));
    const Step s1 = env_step<MODE>(a0.z, a0.w, c0.z, c0.w, player_mask(px, 1), byte_of(cw, 1));
    const Step s2 = env_step<MODE>(a1.x, a1.y, c1.x, c1.y, player_mask(px, 2), byte_of(cw, 2));
    const Step s3 = env_step<MODE>(a1.z, a1.w, c1.z, c1.w, player_mask(px, 3), byte_of(cw, 3));
    o0[2 * i] = make_uint4(s0.lo0, s0.hi0, s1.lo0, s1.hi0);
    o0[2 * i + 1] = make_uint4(s2.lo0, s2.hi0, s3.lo0, s3.hi0);
    o1[2 * i] = make_uint4(s0.lo1, s0.hi1, s1.lo1, s1.hi1);
    o1[2 * i + 1] = make_uint4(s2.lo1, s2.hi1, s3.lo1, s3.hi1);
    // four bytes to a word: a * 2^k + b on the FMA pipe (the fields do not overlap)
    const uint32_t stw = mad_u32(s3.status, 1u << 24, mad_u32(s2.status, 1u << 16, mad_u32(s1.status, 1u << 8, s0.status)));
    opl[i] = pw ^ stw ^ 0x01010101u;  // the side to move changes where the move was made
    olegal[i] = mad_u32(s3.info.legal, 1u << 24, mad_u32(s2.info.legal, 1u << 16, mad_u32(s1.info.legal, 1u << 8, s0.info.legal)));
    oended[i] = mad_u32(s3.info.ended, 1u << 24, mad_u32(s2.info.ended, 1u << 16, mad_u32(s1.info.ended, 1u << 8, s0.info.ended)));
    oreward[i] = make_uint2(mad_u32(s1.info.pair, 1u << 16, s0.info.pair), mad_u32(s3.info.pair, 1u << 16, s2.info.pair));
    ostatus[i] = stw;
}

template <int MODE>
__global__ void __launch_bounds__(256)
k_state_info_h(const uint4 *__restrict__ bb0, const uint4 *__restrict__ bb1, long long quads, uint32_t *olegal, uint32_t *oended,
               uint2 *oreward) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= quads) return;
    const uint4 a0 = bb0[2 * i], a1 = bb0[2 * i + 1], c0 = bb1[2 * i], c1 = bb1[2 * i + 1];
    const c4::h32::Info s0 = c4::h32::state_info<MODE>(a0.x, a0.y, c0.x, c0.y);
    const c4::h32::Info s1 = c4::h32::state_info<MODE>(a0.z, a0.w, c0.z, c0.w);
    const c4::h32::Info s2 = c4::h32::state_info<MODE>(a1.x, a1.y, c1.x, c1.y);
    const c4::h32::Info s3 = c4::h32::state_info<MODE>(a1.z, a1.w, c1.z, c1.w);
    using c4::h32::mad_u32;
    olegal[i] = mad_u32(s3.legal, 1u << 24, mad_u32(s2.legal, 1u << 16, mad_u32(s1.legal, 1u << 8, s0.legal)));
    oended[i] = mad_u32(s3.ended, 1u << 24, mad_u32(s2.ended, 1u << 16, mad_u32(s1.ended, 1u << 8, s0.ended)));
    oreward[i] = make_uint2(mad_u32(s1.pair, 1u << 16, s0.pair), mad_u32(s3.pair, 1u << 16, s2.pair));
}

__global__ void __launch_bounds__(256)
k_state_info(const uint64_t *__restrict__ bb0, const uint64_t *__restrict__ bb1, long long n, uint8_t *olegal,
             uint8_t *oended, int8_t *oreward) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t b0 = bb0[i], b1 = bb1[i];
    const c4::Terminal T = c4::terminal_of(b0, b1);
    if (olegal) olegal[i] = T.ended ? 0 : (uint8_t)c4::legal_mask(b0 | b1);
    if (oended) oended[i] = T.ended ? 1 : 0;
    if (oreward) {
        oreward[2 * i] = T.reward0;
        oreward[2 * i + 1] = (int8_t)-T.reward0;
    }
}

// Left-right mirror of n positions (c4::mirror of both bitboards); flags (may be null = every row): only rows with a non-zero flag
// are mirrored, the others are copied.  Four positions per thread with 16-byte loads / stores of the bitboards and one 32-bit load
// of the flags when `vec` (every pointer 16-byte aligned), else one position per thread.  Each thread reads its positions before it
// writes them, so the output may be the input.
__global__ void __launch_bounds__(256)
k_mirror_states(const uint64_t *bb0, const uint64_t *bb1, const uint8_t *flags, long long n, uint64_t *o0, uint64_t *o1, int vec) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec) {
        if (4 * i + 3 >= n) return;
        const uint4 *v0 = reinterpret_cast<const uint4 *>(bb0) + 2 * i, *v1 = reinterpret_cast<const uint4 *>(bb1) + 2 * i;
        const uint4 a0 = v0[0], a1 = v0[1], c0 = v1[0], c1 = v1[1];
        const uint32_t fw = flags ? reinterpret_cast<const uint32_t *>(flags)[i] : 0x01010101u;
        uint64_t x[4] = {(uint64_t)a0.y << 32 | a0.x, (uint64_t)a0.w << 32 | a0.z, (uint64_t)a1.y << 32 | a1.x, (uint64_t)a1.w << 32 | a1.z};
        uint64_t y[4] = {(uint64_t)c0.y << 32 | c0.x, (uint64_t)c0.w << 32 | c0.z, (uint64_t)c1.y << 32 | c1.x, (uint64_t)c1.w << 32 | c1.z};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool m = ((fw >> (8 * k)) & 0xFFu) != 0u;
            x[k] = m ? c4::mirror(x[k]) : x[k];
            y[k] = m ? c4::mirror(y[k]) : y[k];
        }
        uint4 *w0 = reinterpret_cast<uint4 *>(o0) + 2 * i, *w1 = reinterpret_cast<uint4 *>(o1) + 2 * i;
        w0[0] = make_uint4((uint32_t)x[0], (uint32_t)(x[0] >> 32), (uint32_t)x[1], (uint32_t)(x[1] >> 32));
        w0[1] = make_uint4((uint32_t)x[2], (uint32_t)(x[2] >> 32), (uint32_t)x[3], (uint32_t)(x[3] >> 32));
        w1[0] = make_uint4((uint32_t)y[0], (uint32_t)(y[0] >> 32), (uint32_t)y[1], (uint32_t)(y[1] >> 32));
        w1[1] = make_uint4((uint32_t)y[2], (uint32_t)(y[2] >> 32), (uint32_t)y[3], (uint32_t)(y[3] >> 32));
        return;
    }
    if (i >= n) return;
    const uint64_t b0 = bb0[i], b1 = bb1[i];
    const bool m = !flags || flags[i] != 0;
    o0[i] = m ? c4::mirror(b0) : b0;
    o1[i] = m ? c4::mirror(b1) : b1;
}

// One row of the legal-only softmax (models/games/connect4/model.py:29-35), fp32; x[] in, priors out (0 on illegal columns).
__device__ __forceinline__ void masked_softmax_row(float (&x)[7], uint32_t lg) {
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < 7; ++c)
        if ((lg >> c) & 1u) m = fmaxf(m, x[c]);
    float sum = 0.0f;
#pragma unroll
    for (int c = 0; c < 7; ++c) {
        x[c] = ((lg >> c) & 1u) ? expf(x[c] - m) : 0.0f;
        sum += x[c];
    }
#pragma unroll
    for (int c = 0; c < 7; ++c) x[c] = ((lg >> c) & 1u) ? __fdiv_rn(x[c], sum) : 0.0f;
}

__global__ void __launch_bounds__(256)
k_masked_softmax(const float *__restrict__ logits, const uint8_t *__restrict__ legal, long long n, float *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t lg = legal[i] & 0x7Fu;
    float x[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) x[c] = logits[i * 7 + c];
    masked_softmax_row(x, lg);
#pragma unroll
    for (int c = 0; c < 7; ++c) out[i * 7 + c] = x[c];
}

// Same rows, HBM-coalesced: a row is 28 bytes, so a thread-per-row access pattern touches every 32-byte sector seven times.
// The block's 256 rows (7168 bytes) go through shared memory with 128-bit accesses; rows are read from shared memory at a
// stride of 7 words (odd: conflict-free).  Used for the full 256-row blocks when both arrays are 16-byte aligned; the
// thread-per-row kernel takes the tail.
__global__ void __launch_bounds__(256)
k_masked_softmax_tile(const float4 *__restrict__ logits, const uint8_t *__restrict__ legal, float4 *out) {
    __shared__ float4 tile[448];  // 256 rows x 7 floats
    const size_t b4 = (size_t)blockIdx.x * 448;
    const int t = threadIdx.x;
    tile[t] = logits[b4 + t];
    if (t < 192) tile[256 + t] = logits[b4 + 256 + t];
    const uint32_t lg = legal[(size_t)blockIdx.x * 256 + t] & 0x7Fu;
    __syncthreads();
    float *row = reinterpret_cast<float *>(tile) + 7 * t;
    float x[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) x[c] = row[c];
    masked_softmax_row(x, lg);
#pragma unroll
    for (int c = 0; c < 7; ++c) row[c] = x[c];
    __syncthreads();
    out[b4 + t] = tile[t];
    if (t < 192) out[b4 + 256 + t] = tile[256 + t];
}

// ------------------------------------------------------------------------------------------------
// Counter-based random numbers of the self-play options: Philox4x32-10 (root noise, playout cap randomization)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ double u01_open(uint32_t x) { return ((double)x + 0.5) * 0x1p-32; }  // (0, 1)

// Playout cap randomization (az_set_playout_cap; KataGo): each search of a self-play move step is "full" with probability p_full,
// else "fast".  A full search runs S new simulations, a fast one fast_sims; with visit_budget the search tops the root up to that
// many visits instead, at least one new simulation (n = max(S_t - N_start, 1)).  budget[t] = N_start + n is the root visit count at
// which tree t stops: the BUDGET builds of the selection kernels and of k_run_sims leave it idle from there on.  Only full searches
// become training samples.  The flag of (slot, move step) is a pure function of (seed, global slot, step): Philox keyed by the
// seed, counter {global slot lo, hi, step, CAP_TAG}, full iff u01_open(x) < p_full in fp64 - root noise's counters end in
// column << 24 | attempt < 7 << 24, so the two never share a counter.
constexpr uint32_t CAP_TAG = 0xC0000000u;
// Per-slot counters of the mode, [E][CS_N] u64.
enum { CS_FULL, CS_FAST, CS_RECORDED, CS_DROPPED, CS_N };

struct CapArgs {
    uint32_t *budget;             // [E] absolute root visit count at which the tree stops
    uint8_t *full;                // [E] 1 = the current search is full
    uint8_t *g_full;              // [E][42] the flag of every ply in the game log
    unsigned long long *cstats;   // [E][CS_N]
    unsigned long long seed;
    long long slot_offset;
    double p_full;
    int S, fast, visit_budget;
};

__device__ __forceinline__ bool cap_draw_full(const CapArgs &cp, int t, uint32_t step) {
    const unsigned long long g = (unsigned long long)(cp.slot_offset + t);
    const uint4 r = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), step, CAP_TAG),
                                  make_uint2((uint32_t)cp.seed, (uint32_t)(cp.seed >> 32)));
    return u01_open(r.x) < cp.p_full;
}

// the flag and the budget of the search that starts from a root with n_start visits
__device__ __forceinline__ void cap_set(const CapArgs &cp, int t, bool full, uint32_t n_start) {
    const uint32_t st = (uint32_t)(full ? cp.S : cp.fast);
    const uint32_t n = !cp.visit_budget ? st : (st > n_start + 1u ? st - n_start : 1u);
    cp.full[t] = full ? 1 : 0;
    cp.budget[t] = n_start + n;
}

// the draw of move step `step` for every slot < n from the roots as they are (all_full: every search full with S new simulations,
// for az_set_roots and az_advance_roots, which are not self-play)
__global__ void __launch_bounds__(256) k_cap_draw(Arena a, int n, CapArgs cp, uint32_t step, int all_full) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    if (all_full) cp.visit_budget = 0;  // S new simulations, as without the mode, also on a root that kept its subtree
    cap_set(cp, t, all_full || cap_draw_full(cp, t, step), a.M[(size_t)t * a.cap].x);
}

// ------------------------------------------------------------------------------------------------
// roots / results
__global__ void __launch_bounds__(256)
k_set_roots(Arena a, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, uint64_t c0, uint64_t c1,
            int cpl, int n, int clear_logs) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint64_t b0 = bb0 ? bb0[t] : c0, b1 = bb1 ? bb1[t] : c1;
    const int pl = player ? (player[t] & 1) : cpl;
    a.root_bb0[t] = b0;
    a.root_bb1[t] = b1;
    a.root_player[t] = (uint8_t)pl;
    a.tree_err[t] = c4::terminal_of(b0, b1).ended ? AZ_TREE_ROOT_ENDED : AZ_TREE_OK;
    a.leaf_status[t] = AZ_LEAF_IDLE;
    reset_tree(a, t);
    if (clear_logs) a.g_len[t] = 0;
}

__global__ void __launch_bounds__(256)
k_root_stats(Arena a, int n, int32_t *child_N, double *child_W, float *child_P, double *root_W, int32_t *root_N,
             uint8_t *legal_out, int32_t *err) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const size_t base = (size_t)t * a.cap;
    const uint32_t cb = a.M[base].z;
    const int terr = a.tree_err[t];
    const uint32_t legal = terr ? 0u : c4::legal_mask(a.root_bb0[t] | a.root_bb1[t]);
    int j = 0;
    for (int c = 0; c < 7; ++c) {
        const bool has = cb != 0 && ((legal >> c) & 1u);
        const size_t idx = base + cb + j;
        if (child_N) child_N[(size_t)t * 7 + c] = has ? (int32_t)a.M[idx].x : 0;
        if (child_W) child_W[(size_t)t * 7 + c] = has ? a.W[idx] : 0.0;
        if (child_P) child_P[(size_t)t * 7 + c] = has ? __uint_as_float(a.M[idx].y) : 0.0f;
        if (has) ++j;
    }
    if (root_W) root_W[t] = a.W[base];
    if (root_N) root_N[t] = (int32_t)a.M[base].x;
    if (legal_out) legal_out[t] = (uint8_t)legal;
    if (err) err[t] = terr;
}

__global__ void __launch_bounds__(256)
k_leaf_info(Arena a, int n, uint64_t *o0, uint64_t *o1, uint8_t *opl, uint8_t *olegal, uint8_t *ostatus) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint8_t st = a.leaf_status[t];
    if (o0) o0[t] = a.leaf_bb0[t];
    if (o1) o1[t] = a.leaf_bb1[t];
    if (opl) opl[t] = a.leaf_player[t];
    if (olegal) olegal[t] = (st == AZ_LEAF_EVAL || st == AZ_LEAF_SERVED) ? (uint8_t)c4::legal_mask(a.leaf_bb0[t] | a.leaf_bb1[t]) : 0;
    if (ostatus) ostatus[t] = st;
}

// ------------------------------------------------------------------------------------------------
// This slot's part of a move step: record the sample, draw and play the move, emit the episode header if the game ended.
// Returns through copy_len / copy_dst the finished game's samples still to be copied into the ring.
// GREEDY (az_set_greedy_from): from ply `greedy_from` of the game on, the move is the most visited root child, the lowest
// column on ties (select_action of deepmind_alphazero_pseudocode.py past num_sampling_moves); earlier plies are sampled.
// REUSE (az_set_subtree_reuse): a game that goes on records the played child's node index in reroot[t] for k_reroot instead of
// resetting the tree; every other slot gets REROOT_NONE.
constexpr uint32_t REROOT_NONE = 0u;  // node 0 is the root, never a played child

// BUDGET (az_set_playout_cap): the ply's flag goes into the game log next to the sample, and a finished game emits only the samples
// of its full searches (ep_len = their number, possibly 0); copy_len stays the number of plies, the copy skips the fast ones.
template <bool GREEDY, bool REUSE, bool BUDGET>
__device__ __forceinline__ void sample_move_slot(const Arena &a, int t, const double *__restrict__ uniforms, uint8_t *finished, int step,
                                                 uint64_t init0, uint64_t init1, int initpl, int greedy_from, int &copy_len,
                                                 long long &copy_dst, uint32_t *reroot, const CapArgs &cp) {
    if (finished) finished[t] = 0;
    if (REUSE) reroot[t] = REROOT_NONE;
    if (a.tree_err[t]) return;
    const size_t base = (size_t)t * a.cap;
    const uint4 rootm = a.M[base];
    const uint32_t cb = rootm.z;
    if (cb == 0) return;  // no search ran on this root
    uint64_t b0 = a.root_bb0[t], b1 = a.root_bb1[t];
    int pl = a.root_player[t];
    const uint32_t legal = c4::legal_mask(b0 | b1);
    const int k = __popc(legal);
    const double denom = (double)((int)rootm.x - 1);  // improved_policy denominator (node.py:27)
    // sample = (state, improved_policy) recorded before the move (episode_generator.py:56-62)
    const int len = a.g_len[t];
    int32_t cnt[7];
    double cdf[7];  // indexed by column (static indexing only: stays in registers)
    double acc = 0.0;
    {
        int j = 0;
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            cnt[c] = 0;
            cdf[c] = 0.0;
            if ((legal >> c) & 1u) {
                const int32_t nc = (int32_t)a.M[base + cb + j].x;
                cnt[c] = nc;
                const double p = __ddiv_rn((double)nc, denom);
                acc = (j == 0) ? p : __dadd_rn(acc, p);  // p.cumsum()
                cdf[c] = acc;
                ++j;
            }
        }
    }
    if (len < MAX_PLIES) {
        const size_t o = (size_t)t * MAX_PLIES + len;
        a.g_bb0[o] = b0;
        a.g_bb1[o] = b1;
        a.g_player[o] = (uint8_t)pl;
#pragma unroll
        for (int c = 0; c < 7; ++c) a.g_counts[o * 7 + c] = cnt[c];
        if (BUDGET) cp.g_full[o] = cp.full[t];
    }
    const int new_len = len + 1;
    if (BUDGET) cp.cstats[(size_t)t * CS_N + (cp.full[t] ? CS_FULL : CS_FAST)] += 1ull;
    int col;
    if (GREEDY && len >= greedy_from) {
        int32_t best = -1;
        col = 0;
#pragma unroll
        for (int c = 0; c < 7; ++c)
            if (((legal >> c) & 1u) && cnt[c] > best) {  // strict '>': the first maximum
                best = cnt[c];
                col = c;
            }
    } else {
        // np.random.choice(k, p): cdf /= cdf[-1]; idx = searchsorted(cdf, u, side='right') = #{cdf <= u}
        const double u = uniforms[t];
        const double last = acc;
        int idx = 0;
#pragma unroll
        for (int c = 0; c < 7; ++c)
            if (((legal >> c) & 1u) && __ddiv_rn(cdf[c], last) <= u) ++idx;
        if (idx >= k) idx = k - 1;
        col = c4::nth_legal_column(legal, idx);
    }
    const uint64_t bit = c4::drop_bit(b0 | b1, col);
    if (pl == 0) b0 |= bit; else b1 |= bit;
    const bool win = c4::has4(pl ? b1 : b0);
    const bool ended = win || c4::is_full(b0 | b1);
    uint32_t *st = a.tstats + (size_t)t * NSTAT;
    st[4] += 1u;
    if (!ended) {
        a.root_bb0[t] = b0;
        a.root_bb1[t] = b1;
        a.root_player[t] = (uint8_t)(pl ^ 1);
        a.g_len[t] = new_len;
    } else {
        // outcome to every sample (episode.py:52-54); emit; recycle the slot (episode_generator.py:71-78)
        const int8_t r0 = win ? (pl == 0 ? 1 : -1) : 0;
        int rec = new_len;  // samples the game emits: with the playout cap, its full plies
        if (BUDGET) {
            rec = 0;
            for (int q = 0; q < new_len && q < MAX_PLIES; ++q) rec += cp.g_full[(size_t)t * MAX_PLIES + q];
        }
        const unsigned long long e = atomicAdd(&a.ring[0], 1ull);
        const unsigned long long o = atomicAdd(&a.ring[1], (unsigned long long)rec);
        if ((long long)e < a.ep_cap && (long long)(o + rec) <= a.s_cap) {
            a.ep_slot[e] = t;
            a.ep_step[e] = step;
            a.ep_len[e] = rec;
            a.ep_offset[e] = (int64_t)o;
            a.ep_outcome[2 * e] = r0;
            a.ep_outcome[2 * e + 1] = (int8_t)-r0;
            copy_len = BUDGET && rec == 0 ? 0 : new_len;  // the samples are copied by the whole warp below
            copy_dst = (long long)o;
        } else {
            atomicAdd(&a.ring[2], 1ull);
        }
        if (BUDGET) {
            cp.cstats[(size_t)t * CS_N + CS_RECORDED] += (unsigned long long)rec;
            cp.cstats[(size_t)t * CS_N + CS_DROPPED] += (unsigned long long)(new_len - rec);
        }
        st[5] += 1u;
        a.root_bb0[t] = init0;
        a.root_bb1[t] = init1;
        a.root_player[t] = (uint8_t)initpl;
        a.g_len[t] = 0;
        if (finished) finished[t] = 1;
    }
    if (REUSE && !ended) reroot[t] = cb + (uint32_t)__popc(legal & ((1u << col) - 1u));
    else reset_tree(a, t);  // no subtree reuse: the new root has no children (node.py:37-41)
}

// self-play move step (episode_generator.py:53-78, node.py:23-42): one thread per slot for the move itself; the samples of
// games that ended (up to 42 x 45 bytes each, cold in L2 / HBM) are then copied into the ring by the whole warp, one
// lane per sample, so the few threads with a finished game do not serialise dozens of dependent loads.
// `reroot` and `cp` are trailing arguments read by the REUSE / BUDGET builds only, so the other builds keep the parameter layout.
// BUDGET without REUSE also draws the flag of the slot's next search (step + 1) and writes its budget; with REUSE k_cap_draw does
// that after k_reroot has fixed the new root's visit count.
template <bool GREEDY, bool REUSE, bool BUDGET>
__global__ void __launch_bounds__(128)
k_sample_moves(Arena a, int n, const double *__restrict__ uniforms, uint8_t *finished, int step, uint64_t init0,
               uint64_t init1, int initpl, int greedy_from, uint32_t *reroot, CapArgs cp) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int copy_len = 0;
    long long copy_dst = 0;
    if (t < n) {
        sample_move_slot<GREEDY, REUSE, BUDGET>(a, t, uniforms, finished, step, init0, init1, initpl, greedy_from, copy_len, copy_dst,
                                                reroot, cp);
        if (BUDGET && !REUSE) cap_set(cp, t, cap_draw_full(cp, t, (uint32_t)step + 1u), a.M[(size_t)t * a.cap].x);
    }
    __syncwarp();  // the sample recorded by this step is visible to the lanes that copy it
    unsigned todo = __ballot_sync(FULL, copy_len > 0);
    while (BUDGET && todo) {  // the full plies only, in order: a ballot over the flags, then the ranks
        const int src_lane = __ffs(todo) - 1;
        todo &= todo - 1;
        const int len = __shfl_sync(FULL, copy_len, src_lane);
        const long long dst = __shfl_sync(FULL, copy_dst, src_lane);
        const size_t g0 = (size_t)(t - lane + src_lane) * MAX_PLIES;
        long long rank = dst;
        for (int q0 = 0; q0 < len; q0 += 32) {
            const int q = q0 + lane;
            const bool f = q < len && cp.g_full[g0 + q] != 0;
            const unsigned m = __ballot_sync(FULL, f);
            if (f) {
                const long long d = rank + __popc(m & ((1u << lane) - 1u));
                a.s_bb0[d] = a.g_bb0[g0 + q];
                a.s_bb1[d] = a.g_bb1[g0 + q];
                a.s_player[d] = a.g_player[g0 + q];
#pragma unroll
                for (int i = 0; i < 7; ++i) a.s_counts[d * 7 + i] = a.g_counts[(g0 + q) * 7 + i];
            }
            rank += __popc(m);
        }
    }
    while (!BUDGET && todo) {
        const int src_lane = __ffs(todo) - 1;
        todo &= todo - 1;
        const int len = __shfl_sync(FULL, copy_len, src_lane);
        const long long dst = __shfl_sync(FULL, copy_dst, src_lane);
        const size_t g0 = (size_t)(t - lane + src_lane) * MAX_PLIES;
        for (int q = lane; q < len; q += 32) {
            a.s_bb0[dst + q] = a.g_bb0[g0 + q];
            a.s_bb1[dst + q] = a.g_bb1[g0 + q];
            a.s_player[dst + q] = a.g_player[g0 + q];
        }
        for (int i = lane; i < len * 7; i += 32) a.s_counts[dst * 7 + i] = a.g_counts[g0 * 7 + i];
    }
}

// ------------------------------------------------------------------------------------------------
// Subtree reuse (az_set_subtree_reuse / az_advance_roots): after the move to child c, the subtree of c becomes the tree when c is
// expanded and N(c) + S <= V (max_root_visits), so that the next S simulations keep every visit count <= V and the tree within
// 1 + 7 V nodes.  Otherwise the tree is a fresh root (c never expanded: "fresh"; over the bound: "dropped").
// Per-slot counters of the outcomes, kept apart from tstats: [E][RS_N] u64.
enum { RS_RETAINED, RS_FRESH, RS_DROPPED, RS_NODES, RS_VISITS, RS_N };
constexpr int AZ_MAX_ROOT_VISITS = 1 << 16;  // k_reroot's two bitmaps of 1 + 7 V bits stay within one block's shared memory (115 KB)

// One warp per tree compacts the subtree of c in place.  A node's children always lie above it (first_child > i) and a children
// block is contiguous, so one ascending pass marks the subtree and the retained nodes move down in ascending order (each destination
// is <= its source and below every source not yet read): children blocks stay contiguous and in column order, c becomes node 0
// with {N(c), prior 0, first child remapped} and W(c).  Shared memory: two bitmaps of `words` 32-bit words - the block starts
// (first_child values of every node; a block ends at the next start, at most 7 nodes on, or at `used`), reused for the retained
// count below each word once the subtree is marked, and the subtree membership.
__global__ void __launch_bounds__(32)
k_reroot(Arena a, int n, int S, int V, const uint32_t *__restrict__ reroot, unsigned long long *__restrict__ rstats, int words) {
    extern __shared__ uint32_t smw[];
    uint32_t *start = smw;
    uint32_t *member = smw + words;
    const int t = blockIdx.x;
    const int lane = threadIdx.x;
    if (t >= n) return;
    const uint32_t c = reroot[t];
    if (c == REROOT_NONE) return;
    const size_t base = (size_t)t * a.cap;
    double *__restrict__ W = a.W + base;
    uint4 *__restrict__ M = a.M + base;
    const uint4 mc = M[c];
    unsigned long long *st = rstats + (size_t)t * RS_N;
    if (mc.z == 0 || mc.x + (uint32_t)S > (uint32_t)V) {
        if (lane == 0) {
            reset_tree(a, t);
            st[mc.z == 0 ? RS_FRESH : RS_DROPPED] += 1ull;
        }
        return;
    }
    const uint32_t used = a.used[t];
    for (int w = lane; w < words; w += 32) {
        start[w] = 0u;
        member[w] = 0u;
    }
    __syncwarp();
    for (uint32_t i = lane; i < used; i += 32) {
        const uint32_t cb = reinterpret_cast<const uint32_t *>(M + i)[2];
        if (cb) atomicOr(&start[cb >> 5], 1u << (cb & 31));
    }
    if (lane == 0) atomicOr(&member[c >> 5], 1u << (c & 31));
    __syncwarp();
    // mark: a chunk of 32 nodes may hold a node and its children (then the loop goes round again for them)
    for (uint32_t i0 = c & ~31u; i0 < used; i0 += 32) {
        const uint32_t i = i0 + lane;
        const bool in = i >= c && i < used;
        const uint32_t cb = in ? reinterpret_cast<const uint32_t *>(M + i)[2] : 0u;
        bool done = false;
        for (;;) {
            const bool m = in && ((member[i0 >> 5] >> lane) & 1u);
            if (m && !done && cb) {
                const uint32_t wi = cb >> 5;
                uint64_t win = start[wi];
                if (wi + 1 < (uint32_t)words) win |= (uint64_t)start[wi + 1] << 32;
                const uint64_t after = (win >> (cb & 31)) >> 1;  // block starts at cb + 1, cb + 2, ...
                uint32_t k = after ? (uint32_t)__ffsll((long long)after) : 7u;
                k = k < 7u ? k : 7u;
                k = cb + k <= used ? k : used - cb;
                const uint64_t bits = ((1ull << k) - 1ull) << (cb & 31);
                atomicOr(&member[wi], (uint32_t)bits);
                if (bits >> 32) atomicOr(&member[wi + 1], (uint32_t)(bits >> 32));
            }
            done = done || m;
            __syncwarp();
            if (!__any_sync(FULL, in && !done && ((member[i0 >> 5] >> lane) & 1u))) break;
        }
    }
    __syncwarp();
    // start[w] := retained nodes in words below w (words below c's hold none)
    uint32_t carry = 0;
    const uint32_t wend = (used + 31) >> 5;
    for (uint32_t wb = c >> 5; wb < wend; wb += 32) {
        const uint32_t w = wb + lane;
        const uint32_t cnt = w < wend ? (uint32_t)__popc(member[w]) : 0u;
        uint32_t incl = cnt;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t o = __shfl_up_sync(FULL, incl, off);
            incl += lane >= off ? o : 0u;
        }
        if (w < wend) start[w] = carry + incl - cnt;
        carry += __shfl_sync(FULL, incl, 31);
    }
    __syncwarp();
    // move: node i goes to its rank among the retained nodes
    for (uint32_t i0 = c & ~31u; i0 < used; i0 += 32) {
        const uint32_t i = i0 + lane;
        const uint32_t mw = member[i0 >> 5];
        const bool m = i < used && ((mw >> lane) & 1u);
        double w = 0.0;
        uint4 rec = make_uint4(0u, 0u, 0u, 0u);
        if (m) {
            w = W[i];
            rec = M[i];
            if (rec.z) rec.z = start[rec.z >> 5] + (uint32_t)__popc(member[rec.z >> 5] & ((1u << (rec.z & 31)) - 1u));
            if (i == c) rec.y = 0u;  // the root's prior
        }
        const uint32_t dst = start[i0 >> 5] + (uint32_t)__popc(mw & ((1u << lane) - 1u));
        __syncwarp();  // every source of this chunk is read before any destination of it is written
        if (m) {
            W[dst] = w;
            M[dst] = rec;
        }
    }
    if (lane == 0) {
        a.used[t] = carry;
        st[RS_RETAINED] += 1ull;
        st[RS_NODES] += carry;
        st[RS_VISITS] += mc.x;
    }
}

// az_advance_roots: plays cols[t] on every active root.  An illegal column (or a root in error) leaves the slot untouched; a move
// that ends the game makes that position the root of a fresh tree flagged AZ_TREE_ROOT_ENDED; otherwise k_reroot applies the
// retention rule to the played child (an unexpanded root just gets the new position).  Game logs are not touched.
__global__ void __launch_bounds__(256)
k_advance_roots(Arena a, int n, const uint8_t *__restrict__ cols, uint8_t *__restrict__ status, uint32_t *__restrict__ reroot) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    reroot[t] = REROOT_NONE;
    uint64_t b0 = a.root_bb0[t], b1 = a.root_bb1[t];
    const int pl = a.root_player[t];
    const uint32_t legal = a.tree_err[t] ? 0u : c4::legal_mask(b0 | b1);
    const int col = cols[t];
    if (col >= c4::W || !((legal >> col) & 1u)) {
        status[t] = 1;
        return;
    }
    status[t] = 0;
    const uint32_t cb = a.M[(size_t)t * a.cap].z;
    const uint64_t bit = c4::drop_bit(b0 | b1, col);
    if (pl == 0) b0 |= bit; else b1 |= bit;
    const bool ended = c4::has4(pl ? b1 : b0) || c4::is_full(b0 | b1);
    a.root_bb0[t] = b0;
    a.root_bb1[t] = b1;
    a.root_player[t] = (uint8_t)(pl ^ 1);
    a.leaf_status[t] = AZ_LEAF_IDLE;
    if (ended) a.tree_err[t] = AZ_TREE_ROOT_ENDED;
    if (ended || cb == 0) reset_tree(a, t);
    else reroot[t] = cb + (uint32_t)__popc(legal & ((1u << col) - 1u));
}

__global__ void __launch_bounds__(256) k_reset_trees(Arena a, int n) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) reset_tree(a, t);
}

// ------------------------------------------------------------------------------------------------
// Dirichlet noise on the root priors (az_set_root_noise / az_apply_root_noise; add_exploration_noise of
// deepmind_alphazero_pseudocode.py).  η of a tree is a pure function of (seed, global slot, draw number, column): Philox4x32-10
// keyed by the seed, counter {global slot lo, hi, draw, column << 24 | attempt}, so a sharded run draws what the unsharded run
// draws for the same games.  Gamma variates by Marsaglia-Tsang, every attempt of the rejection loop on its own counter; for
// alpha < 1 in log space, log G(alpha + 1) + log(U) / alpha, normalised with a max-subtracted exp, so that a small alpha cannot
// underflow every component to 0.
constexpr int NOISE_MAX_ATTEMPTS = 1 << 16;  // acceptance is >= 95 % per attempt: never reached in practice

// log of a Gamma(alpha, 1) variate
__device__ double log_gamma_variate(double alpha, uint2 key, uint4 ctr) {
    const bool boost = alpha < 1.0;
    const double d = (boost ? alpha + 1.0 : alpha) - 1.0 / 3.0;
    const double cc = 1.0 / sqrt(9.0 * d);
    double lg = log(d), ub = 0.5;
    for (uint32_t attempt = 0; attempt < (uint32_t)NOISE_MAX_ATTEMPTS; ++attempt) {
        const uint4 r = philox4x32_10(make_uint4(ctr.x, ctr.y, ctr.z, ctr.w | attempt), key);
        const double x = sqrt(-2.0 * log(u01_open(r.x))) * cospi(2.0 * u01_open(r.y));  // Box-Muller
        double v = 1.0 + cc * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        if (log(u01_open(r.z)) < 0.5 * x * x + d - d * v + d * log(v)) {
            lg = log(d * v);
            ub = u01_open(r.w);  // not part of the acceptance test: an independent uniform
            break;
        }
    }
    return boost ? lg + log(ub) / alpha : lg;
}

// eight lanes per tree, lane c < 7 = column c.  Trees in error or without children (the first simulation did not expand the
// root) are left alone; their η rows, and those of inactive slots, are 0.
// BUDGET (az_set_playout_cap): fast searches (full[t] == 0, a trailing argument) get no noise either.
template <bool BUDGET>
__global__ void __launch_bounds__(256)
k_root_noise(Arena a, int n_active, double alpha, float fraction, unsigned long long seed, long long slot_offset, uint32_t draw,
             float *__restrict__ eta, const uint8_t *full) {
    const int t = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const int c = threadIdx.x & 7;
    const int tt = t < a.E ? t : 0;
    const size_t base = (size_t)tt * a.cap;
    const uint32_t cb = a.M[base].z;
    const bool act = t < n_active && a.tree_err[tt] == 0 && cb != 0 && (!BUDGET || full[tt] != 0);
    const uint32_t legal = act ? c4::legal_mask(a.root_bb0[tt] | a.root_bb1[tt]) : 0u;
    const bool mine = c < 7 && ((legal >> c) & 1u);
    double lg = -INFINITY;
    if (mine) {
        const unsigned long long g = (unsigned long long)(slot_offset + t);
        const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
        lg = log_gamma_variate(alpha, key, make_uint4((uint32_t)g, (uint32_t)(g >> 32), draw, (uint32_t)c << 24));
    }
    double m = lg;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) m = fmax(m, __shfl_xor_sync(FULL, m, off));
    const double e = mine ? exp(lg - m) : 0.0;
    double s = e;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) s += __shfl_xor_sync(FULL, s, off);
    const float h = mine ? (float)(e / s) : 0.0f;
    if (mine) {
        // P' = RN(RN(RN(1 - eps) * P) + RN(eps * eta)), fp32, one rounding per operation
        uint32_t *py = reinterpret_cast<uint32_t *>(a.M + base + cb + __popc(legal & ((1u << c) - 1u))) + 1;
        const float p = __uint_as_float(*py);
        *py = __float_as_uint(__fadd_rn(__fmul_rn(__fsub_rn(1.0f, fraction), p), __fmul_rn(fraction, h)));
    }
    if (t < a.E && c < 7) eta[(size_t)t * 7 + c] = h;
}

__global__ void __launch_bounds__(256) k_init_tables(double *rcp, double *sqt, double2 *t2, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rcp[i] = i ? __drcp_rn((double)i) : 0.0;
    sqt[i] = __dsqrt_rn((double)i);
    t2[i] = make_double2(__drcp_rn((double)(i + 1)), __dsqrt_rn((double)i));
}

__global__ void __launch_bounds__(256)
k_export_tree(Arena a, int slot, double *W, uint32_t *N, float *P, uint32_t *CB) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.cap) return;
    const size_t idx = (size_t)slot * a.cap + i;
    const uint4 m = a.M[idx];
    if (W) W[i] = a.W[idx];
    if (N) N[i] = m.x;
    if (P) P[i] = __uint_as_float(m.y);
    if (CB) CB[i] = m.z;
}

// self-test of div_tab against the IEEE division: x = a random double built from the counter, d = 1 .. tab_n-1
__global__ void __launch_bounds__(256)
k_selftest_div(const double *__restrict__ rcp, int tab_n, unsigned long long seed, long long n, unsigned long long *mismatch) {
    unsigned long long bad = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const uint64_t h = azeval::mix64(seed + (uint64_t)i);
        const uint32_t d = 1u + (uint32_t)((h >> 40) % (uint32_t)(tab_n - 1));
        double x;
        switch (h & 3u) {
            case 0: x = __longlong_as_double((long long)((h >> 2) & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ll) * (double)(1u + (uint32_t)((h >> 54) & 255u)); break;  // [1,2) * small int
            case 1: x = (double)(float)__longlong_as_double((long long)((azeval::mix64(h) >> 12) | 0x3FF0000000000000ll)) * (double)d; break;  // fp32 value times d
            case 2: x = (double)(long long)(h >> 33) * (1.0 / 128.0); break;  // dyadic sums (hash evaluator values)
            default: x = __longlong_as_double((long long)((azeval::mix64(h ^ 0x55ull) >> 12) | 0x3FE0000000000000ll)) * __dsqrt_rn((double)(1u + (uint32_t)((h >> 20) & 1023u))); break;  // prior * sqrt(N)
        }
        if ((h >> 63) & 1ull) x = -x;
        if (div_tab(x, d, rcp) != __ddiv_rn(x, (double)d)) ++bad;
    }
    if (bad) atomicAdd(mismatch, bad);
}

__global__ void __launch_bounds__(256) k_sum_stats(const uint32_t *__restrict__ tstats, int E, unsigned long long *tot) {
    unsigned long long loc[NSTAT] = {};
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < E; t += gridDim.x * blockDim.x)
        for (int q = 0; q < NSTAT; ++q) loc[q] += tstats[(size_t)t * NSTAT + q];
    for (int q = 0; q < NSTAT; ++q) {
        unsigned long long x = loc[q];
        for (int off = 16; off >= 1; off >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, off);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(&tot[q], x);
    }
}

__global__ void k_add_u32(uint32_t *p, uint32_t v) { *p += v; }

__global__ void __launch_bounds__(256) k_zero_u32(uint32_t *p, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        p[i] = 0u;
}

char g_create_error[512] = "";

}  // namespace

// ==================================================================================================
struct RingPtrs {
    unsigned long long *ring;
    int32_t *ep_slot, *ep_step, *ep_len;
    int64_t *ep_offset;
    int8_t *ep_outcome;
    uint64_t *s_bb0, *s_bb1;
    uint8_t *s_player;
    int32_t *s_counts;
};

struct az_engine {
    az_config cfg;
    Arena a;
    RingPtrs rings[2];
    int active_ring;
    int G;
    int n_active;
    int step;
    int num_sms;
    int force_hot_nodes;  // -1 = automatic
    int last_hot_nodes;
    int sims_done;  // simulations run on the current roots (arena and tables are sized for num_simulations)
    int compact;         // az_set_leaf_compaction: 1 = every selection is followed by k_compact_leaves, 2 = az_expand_backup_select builds the list itself
    bool compact_valid;  // eval_list / eval_count describe the leaves of the last selection
    int cache_log2;      // az_set_eval_cache: 0 = off
    void *cache_mem;
    bool sel_pending;    // a selection's leaves wait for their expansion
    bool cache_sel;      // ... and that selection used the evaluation cache (the expansion must, too)
    uint64_t init0, init1;
    int initpl;
    bool have_init;
    // az_set_root_noise / az_apply_root_noise / az_root_noise_values
    bool noise_on;
    bool noise_applied;  // the current roots were noised already
    double noise_alpha;
    float noise_fraction;
    uint64_t noise_seed;
    int64_t noise_slot_offset;
    uint32_t noise_draws;  // applications since az_set_root_noise: the draw number of the next one
    float *noise_eta;      // [E][7] η of the last application
    int greedy_from;       // az_set_greedy_from: -1 = off
    bool sym;              // az_set_symmetric_eval: selections write canonical leaves (the SYM kernels)
    bool sym_sel;          // ... and the last selection did (leaf_mirror describes its leaves)
    uint8_t *leaf_mirror;  // [E] 1 = the leaf arrays hold the mirror of the leaf the descent reached (allocated with the first az_set_symmetric_eval)
    int reuse_v;               // az_set_subtree_reuse: max_root_visits V, 0 = off (the arena and the tables are sized for V, else for S)
    uint32_t *reroot;          // [E] played child for k_reroot (REROOT_NONE = nothing to keep); allocated with the first az_set_subtree_reuse
    unsigned long long *rstats;  // [E][RS_N] k_reroot's counters
    bool cap_on;                 // az_set_playout_cap: self-play searches run to per-tree budgets (the BUDGET kernels)
    CapArgs cap;                 // its arrays (allocated with the first az_set_playout_cap) and configuration, as the kernels take them
    int64_t bytes;
    int64_t launches;
    unsigned long long *d_tot;   // [16] stats totals (device)
    unsigned long long acc_tot[NSTAT];  // totals folded on the host across resets
    void *allocs[96];
    int n_allocs;
    char err[512];
};

namespace {

int fail(az_engine *h, int code, const char *fmt, const char *detail) {
    if (h) snprintf(h->err, sizeof h->err, fmt, detail);
    else snprintf(g_create_error, sizeof g_create_error, fmt, detail);
    return code;
}

#define AZ_CUDA(h, call)                                                            \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if (e_ != cudaSuccess) return fail((h), AZ_E_CUDA, #call ": %s", cudaGetErrorString(e_)); \
    } while (0)

static int env_int(const char *name, int dflt) {
    const char *e = getenv(name);
    return e ? atoi(e) : dflt;
}

#define AZ_LAUNCH_CHECK(h, name)                                                    \
    do {                                                                            \
        cudaError_t e_ = cudaGetLastError();                                        \
        if (e_ != cudaSuccess) return fail((h), AZ_E_CUDA, name " launch: %s", cudaGetErrorString(e_)); \
        (h)->launches++;                                                            \
    } while (0)

template <typename T>
int dev_alloc(az_engine *h, T **p, size_t count) {
    void *q = nullptr;
    const size_t bytes = (count ? count : 1) * sizeof(T);
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(h, AZ_E_NOMEM, "cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    if (h->n_allocs >= 96) return fail(h, AZ_E_INVALID, "%s", "allocation table full");
    h->allocs[h->n_allocs++] = q;
    h->bytes += (int64_t)bytes;
    *p = (T *)q;
    return AZ_OK;
}

// releases an allocation of dev_alloc (`bytes` = what it took)
void dev_free(az_engine *h, void *p, size_t bytes) {
    for (int i = 0; i < h->n_allocs; ++i)
        if (h->allocs[i] == p) {
            cudaFree(p);
            h->allocs[i] = h->allocs[--h->n_allocs];
            h->bytes -= (int64_t)bytes;
            return;
        }
}

void use_ring(az_engine *h, int r) {
    const RingPtrs &g = h->rings[r];
    Arena &a = h->a;
    a.ring = g.ring; a.ep_slot = g.ep_slot; a.ep_step = g.ep_step; a.ep_len = g.ep_len; a.ep_offset = g.ep_offset;
    a.ep_outcome = g.ep_outcome; a.s_bb0 = g.s_bb0; a.s_bb1 = g.s_bb1; a.s_player = g.s_player; a.s_counts = g.s_counts;
    h->active_ring = r;
}

inline cudaStream_t S(void *s) { return (cudaStream_t)s; }
inline int blocks_for(long long n, int per_block) { return (int)((n + per_block - 1) / per_block); }

int set_device(az_engine *h) {
    AZ_CUDA(h, cudaSetDevice(h->cfg.device));
    return AZ_OK;
}

}  // namespace

namespace {
int launch_encode(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, const uint8_t *status,
                  long long n, void *out, int layout, cudaStream_t st) {
    if ((reinterpret_cast<uintptr_t>(out) & 15u) != 0) return fail(h, AZ_E_INVALID, "%s", "plane output buffer must be 16-byte aligned");
    const int W = layout_words(layout);
    const int B = (W <= 63) ? 128 : 64;
    const int WP = (W % 2 == 0) ? W + 1 : W;
    const size_t smem = (size_t)B * WP * sizeof(uint32_t);
    const int blocks = blocks_for(n, B);
    uint32_t *o = static_cast<uint32_t *>(out);
    switch (layout) {
        case AZ_LAYOUT_GRID_F32: k_encode<AZ_LAYOUT_GRID_F32><<<blocks, B, smem, st>>>(bb0, bb1, player, status, n, o); break;
        case AZ_LAYOUT_PLANES_F32: k_encode<AZ_LAYOUT_PLANES_F32><<<blocks, B, smem, st>>>(bb0, bb1, player, status, n, o); break;
        case AZ_LAYOUT_PLANES_BF16: k_encode<AZ_LAYOUT_PLANES_BF16><<<blocks, B, smem, st>>>(bb0, bb1, player, status, n, o); break;
        default: k_encode<AZ_LAYOUT_PLANES_BF16_NHWC><<<blocks, B, smem, st>>>(bb0, bb1, player, status, n, o); break;
    }
    AZ_LAUNCH_CHECK(h, "k_encode");
    return AZ_OK;
}

// the playout cap's flags and budgets of every slot for move step `step`, from the roots as they are (all_full: every search full)
int launch_cap_draw(az_engine *h, uint32_t step, bool all_full, cudaStream_t st) {
    k_cap_draw<<<blocks_for(h->a.E, 256), 256, 0, st>>>(h->a, h->a.E, h->cap, step, all_full ? 1 : 0);
    AZ_LAUNCH_CHECK(h, "k_cap_draw");
    return AZ_OK;
}

// k_reroot over the first n slots, after k_sample_moves<REUSE> or k_advance_roots wrote h->reroot
int launch_reroot(az_engine *h, int n, cudaStream_t st) {
    const int words = (h->a.cap + 31) / 32;
    const size_t smem = (size_t)2 * words * sizeof(uint32_t);
    if (smem > 48 * 1024) AZ_CUDA(h, cudaFuncSetAttribute(k_reroot, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_reroot<<<n, 32, smem, st>>>(h->a, n, h->cfg.num_simulations, h->reuse_v, h->reroot, h->rstats, words);
    AZ_LAUNCH_CHECK(h, "k_reroot");
    return AZ_OK;
}
}  // namespace

extern "C" {

int32_t az_abi_version(void) { return AZ_ABI_VERSION; }

const char *az_last_error(const az_engine *h) { return h ? h->err : g_create_error; }

int32_t az_create(const az_config *cfg, az_engine **out) {
    if (!cfg || !out) return fail(nullptr, AZ_E_INVALID, "%s", "az_create: null argument");
    *out = nullptr;
    if (cfg->height != 6 || cfg->width != 7 || cfg->count != 4)
        return fail(nullptr, AZ_E_INVALID, "%s", "az_create: only Config(6,7,4) is supported (scripts/train.py:12)");
    if (cfg->num_games < 1 || cfg->num_simulations < 1 || cfg->num_simulations > 1000000)
        return fail(nullptr, AZ_E_INVALID, "%s", "az_create: num_games >= 1 and 1 <= num_simulations <= 1e6 required");
    int G = cfg->lanes_per_tree == 0 ? 8 : cfg->lanes_per_tree;
    if (G != 8 && G != 16 && G != 32) return fail(nullptr, AZ_E_INVALID, "%s", "az_create: lanes_per_tree must be 8, 16 or 32");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, AZ_E_CUDA, "az_create: no CUDA device (%s); this engine has no CPU path",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, AZ_E_INVALID, "%s", "az_create: bad device ordinal");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, cfg->device);
    if (e != cudaSuccess) return fail(nullptr, AZ_E_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, AZ_E_CUDA, "az_create: device is not sm_100 (%s); kernels are built for sm_100a only", prop.name);

    az_engine *h = (az_engine *)calloc(1, sizeof(az_engine));
    if (!h) return fail(nullptr, AZ_E_NOMEM, "%s", "az_create: host allocation failed");
    h->cfg = *cfg;
    h->G = G;
    h->n_active = cfg->num_games;
    h->num_sms = prop.multiProcessorCount;
    h->force_hot_nodes = cfg->hot_nodes_plus1 > 0 ? cfg->hot_nodes_plus1 - 1 : -1;
    e = cudaSetDevice(cfg->device);
    if (e != cudaSuccess) {
        free(h);
        return fail(nullptr, AZ_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    }
    Arena &a = h->a;
    const int E = cfg->num_games;
    a.E = E;
    a.cap = ((1 + 7 * cfg->num_simulations) + 7) & ~7;
    a.ep_cap = 2ll * E + 64;
    a.s_cap = a.ep_cap * MAX_PLIES;
    const size_t nodes = (size_t)E * a.cap;
    int rc = AZ_OK;
#define AL(ptr, count) if (rc == AZ_OK) rc = dev_alloc(h, &(ptr), (size_t)(count))
    AL(a.W, nodes); AL(a.M, nodes);
    double *d_rcp = nullptr, *d_sqt = nullptr;
    double2 *d_t2 = nullptr;
    a.tab_n = cfg->num_simulations + 8;
    AL(d_rcp, a.tab_n); AL(d_sqt, a.tab_n); AL(d_t2, a.tab_n);
    AL(a.root_bb0, E); AL(a.root_bb1, E); AL(a.root_player, E); AL(a.used, E); AL(a.tree_err, E);
    AL(a.leaf_node, E); AL(a.leaf_bb0, E); AL(a.leaf_bb1, E); AL(a.leaf_player, E); AL(a.leaf_status, E + 16);
    AL(a.leaf_depth, E); AL(a.path, (size_t)E * PATH_STRIDE); AL(a.tstats, (size_t)E * NSTAT);
    AL(a.eval_list, E); AL(a.eval_count, 4); AL(a.cache_ctl, 4);
    AL(a.g_bb0, (size_t)E * MAX_PLIES); AL(a.g_bb1, (size_t)E * MAX_PLIES); AL(a.g_player, (size_t)E * MAX_PLIES);
    AL(a.g_counts, (size_t)E * MAX_PLIES * 7); AL(a.g_len, E);
    for (int r = 0; r < 2; ++r) {
        RingPtrs &g = h->rings[r];
        AL(g.ring, 4);
        AL(g.ep_slot, a.ep_cap); AL(g.ep_step, a.ep_cap); AL(g.ep_len, a.ep_cap); AL(g.ep_offset, a.ep_cap);
        AL(g.ep_outcome, a.ep_cap * 2);
        AL(g.s_bb0, a.s_cap); AL(g.s_bb1, a.s_cap); AL(g.s_player, a.s_cap); AL(g.s_counts, a.s_cap * 7);
    }
    AL(h->d_tot, 16);
#undef AL
    if (rc != AZ_OK) {
        snprintf(g_create_error, sizeof g_create_error, "az_create: %s", h->err);
        for (int i = 0; i < h->n_allocs; ++i) cudaFree(h->allocs[i]);
        free(h);
        return rc;
    }
    a.rcp = d_rcp;
    a.sqt = d_sqt;
    a.t2 = d_t2;
    k_init_tables<<<blocks_for(a.tab_n, 256), 256>>>(d_rcp, d_sqt, d_t2, a.tab_n);
    h->launches++;
    cudaMemset(a.tstats, 0, (size_t)E * NSTAT * sizeof(uint32_t));
    cudaMemset(h->rings[0].ring, 0, 4 * sizeof(unsigned long long));
    cudaMemset(h->rings[1].ring, 0, 4 * sizeof(unsigned long long));
    use_ring(h, 0);
    cudaMemset(h->d_tot, 0, 16 * sizeof(unsigned long long));
    cudaMemset(a.g_len, 0, (size_t)E * sizeof(int32_t));
    cudaMemset(a.eval_count, 0, 4 * sizeof(int32_t));
    cudaMemset(a.cache_ctl, 0, 4 * sizeof(uint32_t));
    // every slot starts at the empty board, player 0 (Config.sample_initial_state())
    k_set_roots<<<blocks_for(E, 256), 256>>>(a, nullptr, nullptr, nullptr, 0ull, 0ull, 0, E, 1);
    h->launches++;
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        snprintf(g_create_error, sizeof g_create_error, "az_create: init failed: %s", cudaGetErrorString(e));
        for (int i = 0; i < h->n_allocs; ++i) cudaFree(h->allocs[i]);
        free(h);
        return AZ_E_CUDA;
    }
    h->init0 = 0;
    h->init1 = 0;
    h->initpl = 0;
    h->have_init = true;
    h->greedy_from = -1;
    *out = h;
    return AZ_OK;
}

int32_t az_destroy(az_engine *h) {
    if (!h) return AZ_OK;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (int i = 0; i < h->n_allocs; ++i) cudaFree(h->allocs[i]);
    if (h->cache_mem) cudaFree(h->cache_mem);
    free(h);
    return AZ_OK;
}

int64_t az_device_bytes(const az_engine *h) { return h ? h->bytes : 0; }
int32_t az_device(const az_engine *h) { return h ? h->cfg.device : -1; }
int64_t az_launch_count(const az_engine *h) { return h ? h->launches : 0; }
int32_t az_tree_capacity(const az_engine *h) { return h ? h->a.cap : 0; }

// AZ_RULES_MODE: the 4-in-line test of the vector rules kernels - 0 = right shifts on the ALU pipe; 1 = left shifts, low words on the
// FMA pipe; 2 / 3 / 4 (the default) = also the high words of 1 / 2 / 3 of the four directions (for the A/B).  Identical results
static int rules_mode() {
    static int mode = -2;
    if (mode == -2) mode = env_int("AZ_RULES_MODE", 4);
    return mode;
}

int32_t az_env_step(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, const uint8_t *col,
                    int64_t n, uint64_t *o0, uint64_t *o1, uint8_t *opl, uint8_t *olegal, uint8_t *oended,
                    int8_t *oreward, uint8_t *ostatus, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (n < 0 || (n > 0 && (!bb0 || !bb1 || !player || !col))) return fail(h, AZ_E_INVALID, "%s", "az_env_step: null input");
    if (n == 0) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    const void *ptrs[] = {bb0, bb1, player, col, o0, o1, opl, olegal, oended, oreward, ostatus};
    bool vec = true;
    for (const void *p : ptrs) vec = vec && p && (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
    const long long quads = vec ? n / 4 : 0, head = quads * 4;
    if (quads) {
        const int mode = rules_mode();
#define AZ_ENV_H(M_)                                                                                                                \
    k_env_step_h<M_><<<blocks_for(quads, 256), 256, 0, S(stream)>>>(                                                                \
        reinterpret_cast<const uint4 *>(bb0), reinterpret_cast<const uint4 *>(bb1), reinterpret_cast<const uint32_t *>(player),     \
        reinterpret_cast<const uint32_t *>(col), quads, reinterpret_cast<uint4 *>(o0), reinterpret_cast<uint4 *>(o1),                \
        reinterpret_cast<uint32_t *>(opl), reinterpret_cast<uint32_t *>(olegal), reinterpret_cast<uint32_t *>(oended),              \
        reinterpret_cast<uint2 *>(oreward), reinterpret_cast<uint32_t *>(ostatus))
        if (mode == 0) AZ_ENV_H(0);
        else if (mode == 2) AZ_ENV_H(2);
        else if (mode == 3) AZ_ENV_H(3);
        else if (mode == 1) AZ_ENV_H(1);
        else AZ_ENV_H(4);
#undef AZ_ENV_H
        AZ_LAUNCH_CHECK(h, "k_env_step_h");
    }
    if (head < n) {
#define OFF(p, k) ((p) ? (p) + (k) : (p))
        k_env_step<<<blocks_for(n - head, 256), 256, 0, S(stream)>>>(bb0 + head, bb1 + head, player + head, col + head, n - head,
                                                                OFF(o0, head), OFF(o1, head), OFF(opl, head), OFF(olegal, head),
                                                                OFF(oended, head), OFF(oreward, 2 * head), OFF(ostatus, head));
        AZ_LAUNCH_CHECK(h, "k_env_step");
#undef OFF
    }
    return AZ_OK;
}

int32_t az_state_info(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int64_t n,
                      uint8_t *olegal, uint8_t *oended, int8_t *oreward, void *stream) {
    (void)player;
    if (!h) return AZ_E_INVALID;
    if (n < 0 || (n > 0 && (!bb0 || !bb1))) return fail(h, AZ_E_INVALID, "%s", "az_state_info: null input");
    if (n == 0) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    const void *ptrs[] = {bb0, bb1, olegal, oended, oreward};
    bool vec = true;
    for (const void *p : ptrs) vec = vec && p && (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
    const long long quads = vec ? n / 4 : 0, head = quads * 4;
    if (quads) {
        const int mode = rules_mode();
#define AZ_INFO_H(M_)                                                                                                                      \
    k_state_info_h<M_><<<blocks_for(quads, 256), 256, 0, S(stream)>>>(reinterpret_cast<const uint4 *>(bb0), reinterpret_cast<const uint4 *>(bb1), \
                                                                      quads, reinterpret_cast<uint32_t *>(olegal),                         \
                                                                      reinterpret_cast<uint32_t *>(oended), reinterpret_cast<uint2 *>(oreward))
        if (mode == 0) AZ_INFO_H(0);
        else if (mode == 2) AZ_INFO_H(2);
        else if (mode == 3) AZ_INFO_H(3);
        else if (mode == 1) AZ_INFO_H(1);
        else AZ_INFO_H(4);
#undef AZ_INFO_H
        AZ_LAUNCH_CHECK(h, "k_state_info_h");
    }
    if (head < n) {
#define OFF(p, k) ((p) ? (p) + (k) : (p))
        k_state_info<<<blocks_for(n - head, 256), 256, 0, S(stream)>>>(bb0 + head, bb1 + head, n - head, OFF(olegal, head),
                                                                  OFF(oended, head), OFF(oreward, 2 * head));
        AZ_LAUNCH_CHECK(h, "k_state_info");
#undef OFF
    }
    return AZ_OK;
}

int32_t az_masked_softmax(az_engine *h, const float *logits, const uint8_t *legal, int64_t n, float *out, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (n < 0 || (n > 0 && (!logits || !legal || !out))) return fail(h, AZ_E_INVALID, "%s", "az_masked_softmax: null argument");
    if (n == 0) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    int64_t head = 0;
    if (((uintptr_t)logits | (uintptr_t)out) % 16 == 0 && n >= 256) {
        head = n & ~(int64_t)255;
        k_masked_softmax_tile<<<(unsigned)(head / 256), 256, 0, S(stream)>>>(reinterpret_cast<const float4 *>(logits), legal,
                                                                             reinterpret_cast<float4 *>(out));
        AZ_LAUNCH_CHECK(h, "k_masked_softmax_tile");
    }
    if (head < n) {
        k_masked_softmax<<<blocks_for(n - head, 256), 256, 0, S(stream)>>>(logits + head * 7, legal + head, n - head, out + head * 7);
        AZ_LAUNCH_CHECK(h, "k_masked_softmax");
    }
    return AZ_OK;
}

static int check_layout(az_engine *h, int layout) {
    if (layout < AZ_LAYOUT_GRID_F32 || layout > AZ_LAYOUT_PLANES_BF16_NHWC) return fail(h, AZ_E_INVALID, "%s", "unknown plane layout");
    return AZ_OK;
}

int32_t az_encode_states(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int64_t n,
                         void *out, int32_t layout, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (n < 0 || (n > 0 && (!bb0 || !bb1 || !player || !out))) return fail(h, AZ_E_INVALID, "%s", "az_encode_states: null argument");
    if (int rc = check_layout(h, layout)) return rc;
    if (n == 0) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    return launch_encode(h, bb0, bb1, player, nullptr, n, out, layout, S(stream));
}

int32_t az_reset_games(az_engine *h, uint64_t init_bb0, uint64_t init_bb1, int32_t init_player, void *stream) {
    if (!h) return AZ_E_INVALID;
    if ((init_bb0 & init_bb1) || ((init_bb0 | init_bb1) & ~c4::BOARD) || (init_player != 0 && init_player != 1))
        return fail(h, AZ_E_INVALID, "%s", "az_reset_games: invalid initial position");
    if (int rc = set_device(h)) return rc;
    const int E = h->a.E;
    k_set_roots<<<blocks_for(E, 256), 256, 0, S(stream)>>>(h->a, nullptr, nullptr, nullptr, init_bb0, init_bb1, init_player,
                                                          E, 1);
    AZ_LAUNCH_CHECK(h, "k_set_roots");
    if (h->cap_on)
        if (int rc = launch_cap_draw(h, 0u, false, S(stream))) return rc;
    AZ_CUDA(h, cudaMemsetAsync(h->rings[0].ring, 0, 4 * sizeof(unsigned long long), S(stream)));
    AZ_CUDA(h, cudaMemsetAsync(h->rings[1].ring, 0, 4 * sizeof(unsigned long long), S(stream)));
    h->init0 = init_bb0;
    h->init1 = init_bb1;
    h->initpl = init_player;
    h->have_init = true;
    h->n_active = E;
    h->step = 0;
    h->sims_done = 0;
    h->noise_applied = false;
    h->sel_pending = false;
    return AZ_OK;
}

int32_t az_set_roots(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int32_t n,
                     void *stream) {
    if (!h) return AZ_E_INVALID;
    if (n < 1 || n > h->a.E || !bb0 || !bb1 || !player) return fail(h, AZ_E_INVALID, "%s", "az_set_roots: need 1 <= n <= num_games and non-null positions");
    if (int rc = set_device(h)) return rc;
    k_set_roots<<<blocks_for(n, 256), 256, 0, S(stream)>>>(h->a, bb0, bb1, player, 0ull, 0ull, 0, n, 0);
    AZ_LAUNCH_CHECK(h, "k_set_roots");
    if (h->cap_on)  // not a self-play move step: every search is full
        if (int rc = launch_cap_draw(h, 0u, true, S(stream))) return rc;
    h->n_active = n;
    h->sims_done = 0;
    h->noise_applied = false;
    h->sel_pending = false;
    return AZ_OK;
}

#ifdef AZ_TRUNK_CLOCKS
int32_t az_debug_run_clocks(long long *out, int reset) {
    if (reset) { long long z[8] = {0}; return cudaMemcpyToSymbol(g_run_clk, z, sizeof z) == cudaSuccess ? 0 : 1; }
    return cudaMemcpyFromSymbol(out, g_run_clk, sizeof(g_run_clk)) == cudaSuccess ? 0 : 1;
}
#endif

// Which descend variant a launch of `blocks` 64-thread blocks gets: the latency-optimised one while the grid leaves the SMs
// mostly idle (<= 6 blocks = 12 warps per SM), the throughput one beyond.  AZ_TREE_VARIANT=lat|thr overrides (A/B runs).
static bool latency_variant(const az_engine *h, int blocks) {
    static int forced = -2;
    if (forced == -2) {
        const char *e = getenv("AZ_TREE_VARIANT");
        forced = !e ? -1 : (e[0] == 'l' ? 1 : (e[0] == 't' ? 0 : -1));
    }
    if (forced >= 0) return forced == 1;
    return blocks <= 6 * h->num_sms;
}

static int32_t run_sims_impl(az_engine *h, int32_t num_sims, int32_t eval_kind, const double *uniforms, uint8_t *finished, bool move,
                             void *stream);

int32_t az_run_simulations(az_engine *h, int32_t num_sims, int32_t eval_kind, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (num_sims == 0) return AZ_OK;
    return run_sims_impl(h, num_sims, eval_kind, nullptr, nullptr, false, stream);
}

/* az_run_simulations followed by az_sample_moves in ONE launch (same results): the self-play move step for the built-in
 * evaluators.  uniforms[num_games] f64 in [0,1) (device), finished[num_games] u8 or null. */
int32_t az_run_move_step(az_engine *h, int32_t num_sims, int32_t eval_kind, const double *uniforms, uint8_t *finished, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!uniforms) return fail(h, AZ_E_INVALID, "%s", "az_run_move_step: null uniforms");
    if (!h->have_init) return fail(h, AZ_E_STATE, "%s", "az_run_move_step: call az_reset_games first");
    if (num_sims < 1) return fail(h, AZ_E_INVALID, "%s", "az_run_move_step: num_sims < 1");
    // the greedy rule, subtree reuse and the playout cap live in k_sample_moves (+ k_reroot) only: the search (its hot prefix written
    // back), then the move
    if (h->greedy_from >= 0 || h->reuse_v > 0 || h->cap_on) {
        const int32_t rc = run_sims_impl(h, num_sims, eval_kind, nullptr, nullptr, false, stream);
        if (rc != AZ_OK) return rc;
        return az_sample_moves(h, uniforms, finished, stream);
    }
    const int32_t rc = run_sims_impl(h, num_sims, eval_kind, uniforms, finished, true, stream);
    if (rc != AZ_OK) return rc;
    h->step++;
    h->sims_done = 0;
    h->noise_applied = false;
    return AZ_OK;
}

static int32_t run_sims_impl(az_engine *h, int32_t num_sims, int32_t eval_kind, const double *uniforms, uint8_t *finished, bool move,
                             void *stream) {
    if (num_sims < 0) return fail(h, AZ_E_INVALID, "%s", "az_run_simulations: num_sims < 0");
    if (h->sims_done + num_sims > h->cfg.num_simulations)
        return fail(h, AZ_E_INVALID, "%s", "az_run_simulations: more simulations on these roots than the arena holds (1 + 7*num_simulations nodes per tree)");
    if (eval_kind != AZ_EVAL_UNIFORM && eval_kind != AZ_EVAL_HASH) return fail(h, AZ_E_INVALID, "%s", "az_run_simulations: unknown evaluator");
    if (h->sym) return fail(h, AZ_E_STATE, "%s", "az_run_simulations: the fused built-in path has no symmetric evaluation (az_set_symmetric_eval)");
    if (num_sims == 0) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    const double c = h->cfg.c_puct;
    // hot-node count K: as many as shared memory allows while every block of the grid stays resident
    const int tpw = 32 / h->G, trees_per_block = 2 * tpw;
    const int blocks = blocks_for(n, trees_per_block);
    int per_sm = (blocks + h->num_sms - 1) / h->num_sms;
    if (per_sm > 14) per_sm = 14;  // register-limited residency of 64-thread blocks (80 registers, ncu)
    // hot-node count K: the largest multiple of 8 such that every block of the grid stays resident (228 KB of shared memory per SM,
    // 1 KB of it reserved per resident block; one block may use up to 200 KB) - measured monotonic: more hot nodes, faster
    const long long per_block = (long long)(228 * 1024) / per_sm - 1024;
    // {1/(n+1), sqrt(n)} pairs + 1/n: 24 bytes per entry (19 KB at 800 simulations per move).  The tables go to shared memory
    // whenever they leave at least half of the block's share to the hot nodes: always for S <= 248, and for S = 800 up to
    // 5 resident blocks per SM (<= 5920 trees); denser grids run the throughput variant, where a level's latency matters less.
    const int tabs_in_smem = (long long)h->a.tab_n * 24 <= (per_block < 200 * 1024 ? per_block : 200 * 1024) / 2 ? 1 : 0;
    const size_t tab_bytes = tabs_in_smem ? (size_t)h->a.tab_n * 24 : 0;
    int K = 0;
    {
        const long long budget = (per_block < 200 * 1024 ? per_block : 200 * 1024) - (long long)tab_bytes - (long long)trees_per_block * PATH_STRIDE * 4;
        long long kmax = budget > 0 ? budget / ((long long)trees_per_block * 16) : 0;
        if (kmax > 1024) kmax = 1024;
        if (kmax > h->a.cap) kmax = h->a.cap;
        K = (int)(kmax & ~7ll);
    }
    if (h->force_hot_nodes >= 0) K = (h->force_hot_nodes < h->a.cap ? h->force_hot_nodes : h->a.cap) & ~7;
    if (h->a.cap > 65535) K = 0;  // the 16-byte shared-memory record holds visit count and child index in 16 bits each
    const size_t smem = (size_t)trees_per_block * ((size_t)K * 16 + PATH_STRIDE * 4) + tab_bytes;
    const bool lat = latency_variant(h, blocks);
    MoveArgs mv;
    mv.uniforms = uniforms;
    mv.finished = finished;
    mv.init0 = h->init0;
    mv.init1 = h->init1;
    mv.step = h->step;
    mv.initpl = h->initpl;
    const bool budget = h->cap_on;  // never with `move`: az_run_move_step leaves the move to k_sample_moves then
#define AZ_RUN3(TPW_, EV_, LAT_, MOVE_, TSM_, BUD_)                                                                                               \
    do {                                                                                                                                          \
        AZ_CUDA(h, cudaFuncSetAttribute(k_run_sims<TPW_, EV_, LAT_, MOVE_, TSM_, BUD_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        k_run_sims<TPW_, EV_, LAT_, MOVE_, TSM_, BUD_><<<blocks, 64, smem, S(stream)>>>(h->a, n, num_sims, c, K, mv, h->cap.budget);            \
    } while (0)
#define AZ_RUN2(TPW_, EV_, LAT_, MOVE_, BUD_)                       \
    do {                                                            \
        if (tabs_in_smem) AZ_RUN3(TPW_, EV_, LAT_, MOVE_, true, BUD_); \
        else AZ_RUN3(TPW_, EV_, LAT_, MOVE_, false, BUD_);          \
    } while (0)
#define AZ_RUN1(TPW_, EV_, LAT_)                           \
    do {                                                   \
        if (move) AZ_RUN2(TPW_, EV_, LAT_, true, false);   \
        else if (budget) AZ_RUN2(TPW_, EV_, LAT_, false, true); \
        else AZ_RUN2(TPW_, EV_, LAT_, false, false);       \
    } while (0)
#define AZ_RUN(TPW_, EV_)                  \
    do {                                   \
        if (lat) AZ_RUN1(TPW_, EV_, true); \
        else AZ_RUN1(TPW_, EV_, false);    \
    } while (0)
    if (tpw == 1) {
        if (eval_kind == AZ_EVAL_UNIFORM) AZ_RUN(1, AZ_EVAL_UNIFORM); else AZ_RUN(1, AZ_EVAL_HASH);
    } else if (tpw == 2) {
        if (eval_kind == AZ_EVAL_UNIFORM) AZ_RUN(2, AZ_EVAL_UNIFORM); else AZ_RUN(2, AZ_EVAL_HASH);
    } else {
        if (eval_kind == AZ_EVAL_UNIFORM) AZ_RUN(4, AZ_EVAL_UNIFORM); else AZ_RUN(4, AZ_EVAL_HASH);
    }
#undef AZ_RUN
#undef AZ_RUN1
#undef AZ_RUN2
#undef AZ_RUN3
    h->last_hot_nodes = K;
    h->sims_done += num_sims;
    AZ_LAUNCH_CHECK(h, "k_run_sims");
    return AZ_OK;
}

// The selections probe the evaluation cache while it exists and the evaluator walks the compacted leaf list (the list's kernel, or the
// last warp of k_expand_select<COMPACT>, advances the launch number that tells this launch's claims from earlier ones).
static bool cache_active(const az_engine *h) { return h->a.cache != nullptr && h->compact != 0; }

int32_t az_select_leaves(az_engine *h, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    if (h->sims_done + 1 > h->cfg.num_simulations)
        return fail(h, AZ_E_INVALID, "%s", "az_select_leaves: more simulations on these roots than the arena holds");
    const int tpb = 2 * (32 / h->G);
    const bool lat = latency_variant(h, blocks_for(n, tpb));
    const bool cache = cache_active(h);
    const bool sym = h->sym;
    const bool budget = h->cap_on;
#define AZ_SEL3(TPW_, SYM_, BUD_)                                                                                                        \
    do {                                                                                                                                 \
        if (cache) {                                                                                                                     \
            if (lat) k_select<TPW_, true, true, SYM_, BUD_><<<blocks_for(n, tpb), 64, 0, S(stream)>>>(h->a, n, h->cfg.c_puct, h->leaf_mirror, h->cap.budget);  \
            else k_select<TPW_, false, true, SYM_, BUD_><<<blocks_for(n, tpb), 64, 0, S(stream)>>>(h->a, n, h->cfg.c_puct, h->leaf_mirror, h->cap.budget);     \
        } else {                                                                                                                         \
            if (lat) k_select<TPW_, true, false, SYM_, BUD_><<<blocks_for(n, tpb), 64, 0, S(stream)>>>(h->a, n, h->cfg.c_puct, h->leaf_mirror, h->cap.budget); \
            else k_select<TPW_, false, false, SYM_, BUD_><<<blocks_for(n, tpb), 64, 0, S(stream)>>>(h->a, n, h->cfg.c_puct, h->leaf_mirror, h->cap.budget);    \
        }                                                                                                                                \
    } while (0)
#define AZ_SEL2(TPW_, SYM_)                        \
    do {                                           \
        if (budget) AZ_SEL3(TPW_, SYM_, true);     \
        else AZ_SEL3(TPW_, SYM_, false);           \
    } while (0)
#define AZ_SEL(TPW_)                      \
    do {                                  \
        if (sym) AZ_SEL2(TPW_, true);     \
        else AZ_SEL2(TPW_, false);        \
    } while (0)
    if (h->G == 32) AZ_SEL(1);
    else if (h->G == 16) AZ_SEL(2);
    else AZ_SEL(4);
#undef AZ_SEL
#undef AZ_SEL2
#undef AZ_SEL3
    AZ_LAUNCH_CHECK(h, "k_select");
    h->compact_valid = h->compact != 0;
    if (h->compact) {
        k_compact_leaves<<<1, 1024, 0, S(stream)>>>(h->a.leaf_status, n, h->a.eval_list, h->a.eval_count, env_int("AZ_COMPACT_STAGE", 1),
                                                    cache ? h->a.cache_ctl : nullptr);
        AZ_LAUNCH_CHECK(h, "k_compact_leaves");
    }
    h->sims_done += 1;
    h->sel_pending = true;
    h->cache_sel = cache;
    h->sym_sel = sym;
    return AZ_OK;
}

int32_t az_gather_leaves(az_engine *h, void *out, int32_t layout, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!out) return fail(h, AZ_E_INVALID, "%s", "az_gather_leaves: null output");
    if (int rc = check_layout(h, layout)) return rc;
    if (int rc = set_device(h)) return rc;
    const long long n = h->n_active;
    return launch_encode(h, h->a.leaf_bb0, h->a.leaf_bb1, h->a.leaf_player, h->a.leaf_status, n, out, layout, S(stream));
}

int32_t az_expand_backup(az_engine *h, const float *policy, const float *values, int32_t policy_kind, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!policy || !values) return fail(h, AZ_E_INVALID, "%s", "az_expand_backup: null evaluator output");
    if (policy_kind != AZ_POLICY_LOGITS && policy_kind != AZ_POLICY_PRIORS) return fail(h, AZ_E_INVALID, "%s", "az_expand_backup: bad policy_kind");
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    const bool cache = h->sel_pending && h->cache_sel;  // SERVED leaves and claims exist only after a cached selection
    const bool sym = h->sel_pending && h->sym_sel;      // mirrored leaves exist only after a symmetric selection
#define AZ_EB2(TPW_, SYM_)                                                                                                          \
    do {                                                                                                                            \
        if (cache) k_expand_backup<TPW_, true, SYM_><<<blocks_for(n, 2 * TPW_), 64, 0, S(stream)>>>(h->a, n, policy, values, policy_kind, h->leaf_mirror);  \
        else k_expand_backup<TPW_, false, SYM_><<<blocks_for(n, 2 * TPW_), 64, 0, S(stream)>>>(h->a, n, policy, values, policy_kind, h->leaf_mirror);  \
    } while (0)
#define AZ_EB(TPW_)                      \
    do {                                 \
        if (sym) AZ_EB2(TPW_, true);     \
        else AZ_EB2(TPW_, false);        \
    } while (0)
    if (h->G == 32) AZ_EB(1);
    else if (h->G == 16) AZ_EB(2);
    else AZ_EB(4);
#undef AZ_EB
#undef AZ_EB2
    AZ_LAUNCH_CHECK(h, "k_expand_backup");
    h->compact_valid = false;  // the leaves are consumed
    h->sel_pending = false;
    return AZ_OK;
}

/* az_expand_backup followed by az_select_leaves in ONE launch (same results): between two evaluator calls of the
 * network-in-the-loop simulation loop (search.py:66-91) only this kernel runs. */
int32_t az_expand_backup_select(az_engine *h, const float *policy, const float *values, int32_t policy_kind, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!policy || !values) return fail(h, AZ_E_INVALID, "%s", "az_expand_backup_select: null evaluator output");
    if (policy_kind != AZ_POLICY_LOGITS && policy_kind != AZ_POLICY_PRIORS) return fail(h, AZ_E_INVALID, "%s", "az_expand_backup_select: bad policy_kind");
    if (h->sims_done + 1 > h->cfg.num_simulations)
        return fail(h, AZ_E_INVALID, "%s", "az_expand_backup_select: more simulations on these roots than the arena holds");
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    const int tpb = 2 * (32 / h->G);
    const bool lat = latency_variant(h, blocks_for(n, tpb));
    const bool fused = h->compact == 2;
    const bool cache = cache_active(h);
    if (h->sel_pending && h->cache_sel != cache)
        return fail(h, AZ_E_STATE, "%s", "az_expand_backup_select: the evaluation cache or leaf compaction changed between a selection and its expansion");
    const bool sym = h->sym;  // az_set_symmetric_eval refuses while a selection is pending: the expansion matches its selection
    const bool budget = h->cap_on;
#define AZ_ES4(TPW_, LAT_, CMP_, SYM_, BUD_)                                                                                                \
    do {                                                                                                                              \
        if (cache) k_expand_select<TPW_, LAT_, CMP_, true, SYM_, BUD_><<<blocks_for(n, tpb), 64, 0, S(stream)>>>(h->a, n, policy, values, policy_kind, h->cfg.c_puct, h->leaf_mirror, h->cap.budget);  \
        else k_expand_select<TPW_, LAT_, CMP_, false, SYM_, BUD_><<<blocks_for(n, tpb), 64, 0, S(stream)>>>(h->a, n, policy, values, policy_kind, h->cfg.c_puct, h->leaf_mirror, h->cap.budget);  \
    } while (0)
#define AZ_ES3(TPW_, LAT_, CMP_, SYM_)                   \
    do {                                                 \
        if (budget) AZ_ES4(TPW_, LAT_, CMP_, SYM_, true); \
        else AZ_ES4(TPW_, LAT_, CMP_, SYM_, false);      \
    } while (0)
#define AZ_ES2(TPW_, LAT_, CMP_)                     \
    do {                                             \
        if (sym) AZ_ES3(TPW_, LAT_, CMP_, true);     \
        else AZ_ES3(TPW_, LAT_, CMP_, false);        \
    } while (0)
#define AZ_ES(TPW_)                               \
    do {                                          \
        if (fused) {                              \
            if (lat) AZ_ES2(TPW_, true, true);    \
            else AZ_ES2(TPW_, false, true);       \
        } else {                                  \
            if (lat) AZ_ES2(TPW_, true, false);   \
            else AZ_ES2(TPW_, false, false);      \
        }                                         \
    } while (0)
    if (h->G == 32) AZ_ES(1);
    else if (h->G == 16) AZ_ES(2);
    else AZ_ES(4);
#undef AZ_ES
#undef AZ_ES2
#undef AZ_ES3
#undef AZ_ES4
    AZ_LAUNCH_CHECK(h, "k_expand_select");
    h->compact_valid = h->compact != 0;
    if (h->compact == 1) {
        k_compact_leaves<<<1, 1024, 0, S(stream)>>>(h->a.leaf_status, n, h->a.eval_list, h->a.eval_count, env_int("AZ_COMPACT_STAGE", 1),
                                                    cache ? h->a.cache_ctl : nullptr);
        AZ_LAUNCH_CHECK(h, "k_compact_leaves");
    }
    h->sims_done += 1;
    h->sel_pending = true;
    h->cache_sel = cache;
    h->sym_sel = sym;
    return AZ_OK;
}

int32_t az_leaf_info(az_engine *h, uint64_t *o0, uint64_t *o1, uint8_t *opl, uint8_t *olegal, uint8_t *ostatus,
                     void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    k_leaf_info<<<blocks_for(n, 256), 256, 0, S(stream)>>>(h->a, n, o0, o1, opl, olegal, ostatus);
    AZ_LAUNCH_CHECK(h, "k_leaf_info");
    return AZ_OK;
}

int32_t az_leaf_arrays(az_engine *h, const uint64_t **bb0, const uint64_t **bb1, const uint8_t **status, int32_t *n_active) {
    if (!h) return AZ_E_INVALID;
    if (bb0) *bb0 = h->a.leaf_bb0;
    if (bb1) *bb1 = h->a.leaf_bb1;
    if (status) *status = h->a.leaf_status;
    if (n_active) *n_active = h->n_active;
    return AZ_OK;
}

/* the slots whose leaf waits for the evaluator after the last az_select_leaves / az_expand_backup_select, ascending, and their
 * number - both on the device (engine-owned, valid until az_destroy) */
int32_t az_leaf_compact(az_engine *h, const int32_t **eval_list, const int32_t **eval_count) {
    if (!h) return AZ_E_INVALID;
    if (eval_list) *eval_list = h->compact_valid ? h->a.eval_list : nullptr;
    if (eval_count) *eval_count = h->compact_valid ? h->a.eval_count : nullptr;
    return AZ_OK;
}

int32_t az_set_leaf_compaction(az_engine *h, int32_t on) {
    if (!h) return AZ_E_INVALID;
    if (on < 0 || on > 2) return fail(h, AZ_E_INVALID, "%s", "az_set_leaf_compaction: 0 (off), 1 (one more launch, ascending list) or 2 (fused into az_expand_backup_select)");
    h->compact = on;
    return AZ_OK;
}

int32_t az_leaf_players(az_engine *h, const uint8_t **player) {
    if (!h || !player) return AZ_E_INVALID;
    *player = h->a.leaf_player;
    return AZ_OK;
}

int32_t az_root_stats(az_engine *h, int32_t *child_N, double *child_W, float *child_P, double *root_W, int32_t *root_N,
                      uint8_t *legal, int32_t *err, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    k_root_stats<<<blocks_for(n, 256), 256, 0, S(stream)>>>(h->a, n, child_N, child_W, child_P, root_W, root_N, legal, err);
    AZ_LAUNCH_CHECK(h, "k_root_stats");
    return AZ_OK;
}

int32_t az_export_tree(az_engine *h, int32_t slot, double *W, uint32_t *N, float *P, uint32_t *first_child,
                       int32_t *used_host) {
    if (!h) return AZ_E_INVALID;
    if (slot < 0 || slot >= h->a.E) return fail(h, AZ_E_INVALID, "%s", "az_export_tree: bad slot");
    if (int rc = set_device(h)) return rc;
    AZ_CUDA(h, cudaDeviceSynchronize());
    k_export_tree<<<blocks_for(h->a.cap, 256), 256>>>(h->a, slot, W, N, P, first_child);
    AZ_LAUNCH_CHECK(h, "k_export_tree");
    if (used_host) {
        uint32_t u = 0;
        AZ_CUDA(h, cudaMemcpy(&u, h->a.used + slot, sizeof u, cudaMemcpyDeviceToHost));
        *used_host = (int32_t)u;
    }
    AZ_CUDA(h, cudaDeviceSynchronize());
    return AZ_OK;
}

int32_t az_sample_moves(az_engine *h, const double *uniforms, uint8_t *finished, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!uniforms) return fail(h, AZ_E_INVALID, "%s", "az_sample_moves: null uniforms");
    if (!h->have_init) return fail(h, AZ_E_STATE, "%s", "az_sample_moves: call az_reset_games first");
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    const bool reuse = h->reuse_v > 0;
    const bool budget = h->cap_on;
#define AZ_SM2(G_, R_, B_)                                                                                                         \
    k_sample_moves<G_, R_, B_><<<blocks_for(n, 128), 128, 0, S(stream)>>>(h->a, n, uniforms, finished, h->step, h->init0, h->init1, \
                                                                        h->initpl, G_ ? h->greedy_from : -1, R_ ? h->reroot : nullptr, h->cap)
#define AZ_SM(G_, R_)                  \
    do {                               \
        if (budget) AZ_SM2(G_, R_, true); \
        else AZ_SM2(G_, R_, false);    \
    } while (0)
    if (h->greedy_from >= 0) {
        if (reuse) AZ_SM(true, true);
        else AZ_SM(true, false);
    } else {
        if (reuse) AZ_SM(false, true);
        else AZ_SM(false, false);
    }
#undef AZ_SM
#undef AZ_SM2
    AZ_LAUNCH_CHECK(h, "k_sample_moves");
    if (reuse) {
        if (int rc = launch_reroot(h, n, S(stream))) return rc;
        if (budget)  // the next search's budget counts from the visits the new root kept
            if (int rc = launch_cap_draw(h, (uint32_t)h->step + 1u, false, S(stream))) return rc;
    }
    h->step++;
    h->sims_done = 0;
    h->noise_applied = false;
    return AZ_OK;
}

int32_t az_set_root_noise(az_engine *h, const az_root_noise *cfg) {
    if (!h) return AZ_E_INVALID;
    if (!cfg) {
        h->noise_on = false;
        return AZ_OK;
    }
    if (!(cfg->alpha > 0.0 && cfg->alpha <= 1e6))
        return fail(h, AZ_E_INVALID, "%s", "az_set_root_noise: alpha must be in (0, 1e6]");
    if (!(cfg->fraction >= 0.0f && cfg->fraction <= 1.0f))
        return fail(h, AZ_E_INVALID, "%s", "az_set_root_noise: fraction must be in [0, 1]");
    if (cfg->slot_offset < 0 || cfg->slot_offset > ((int64_t)1 << 62))
        return fail(h, AZ_E_INVALID, "%s", "az_set_root_noise: slot_offset must be in [0, 2^62]");
    if (int rc = set_device(h)) return rc;
    if (!h->noise_eta) {
        if (int rc = dev_alloc(h, &h->noise_eta, (size_t)h->a.E * 7)) return rc;
        AZ_CUDA(h, cudaMemset(h->noise_eta, 0, (size_t)h->a.E * 7 * sizeof(float)));
    }
    h->noise_on = true;
    h->noise_alpha = cfg->alpha;
    h->noise_fraction = cfg->fraction;
    h->noise_seed = cfg->seed;
    h->noise_slot_offset = cfg->slot_offset;
    h->noise_draws = 0;
    return AZ_OK;
}

int32_t az_apply_root_noise(az_engine *h, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!h->noise_on) return fail(h, AZ_E_STATE, "%s", "az_apply_root_noise: no noise configured (az_set_root_noise)");
    if (h->sims_done != 1 || h->sel_pending || h->noise_applied)
        return fail(h, AZ_E_STATE, "%s", "az_apply_root_noise: valid once, after exactly one complete simulation on the current roots");
    if (int rc = set_device(h)) return rc;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    AZ_CUDA(h, cudaStreamIsCapturing(S(stream), &cap));
    if (cap != cudaStreamCaptureStatusNone)
        return fail(h, AZ_E_STATE, "%s", "az_apply_root_noise: not inside a CUDA graph capture (the draw number is a launch argument)");
    const int E = h->a.E;
    if (h->cap_on)
        k_root_noise<true><<<blocks_for((long long)E * 8, 256), 256, 0, S(stream)>>>(h->a, h->n_active, h->noise_alpha, h->noise_fraction,
                                                                                    h->noise_seed, h->noise_slot_offset, h->noise_draws,
                                                                                    h->noise_eta, h->cap.full);
    else
        k_root_noise<false><<<blocks_for((long long)E * 8, 256), 256, 0, S(stream)>>>(h->a, h->n_active, h->noise_alpha, h->noise_fraction,
                                                                                     h->noise_seed, h->noise_slot_offset, h->noise_draws,
                                                                                     h->noise_eta, nullptr);
    AZ_LAUNCH_CHECK(h, "k_root_noise");
    h->noise_draws++;
    h->noise_applied = true;
    return AZ_OK;
}

int32_t az_root_noise_values(az_engine *h, float *eta, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!eta) return fail(h, AZ_E_INVALID, "%s", "az_root_noise_values: null output");
    if (!h->noise_eta) return fail(h, AZ_E_STATE, "%s", "az_root_noise_values: no noise configured (az_set_root_noise)");
    if (int rc = set_device(h)) return rc;
    AZ_CUDA(h, cudaMemcpyAsync(eta, h->noise_eta, (size_t)h->a.E * 7 * sizeof(float), cudaMemcpyDeviceToDevice, S(stream)));
    return AZ_OK;
}

int32_t az_set_greedy_from(az_engine *h, int32_t plies) {
    if (!h) return AZ_E_INVALID;
    h->greedy_from = plies < 0 ? -1 : plies;
    return AZ_OK;
}

static int ring_counts(az_engine *h, int ring, int64_t *ne, int64_t *ns, cudaStream_t st) {
    unsigned long long r[4];
    AZ_CUDA(h, cudaMemcpyAsync(r, h->rings[ring].ring, sizeof r, cudaMemcpyDeviceToHost, st));
    AZ_CUDA(h, cudaStreamSynchronize(st));
    if (ne) *ne = (int64_t)r[0];
    if (ns) *ns = (int64_t)r[1];
    if (r[2]) return fail(h, AZ_E_OVERFLOW, "%s", "episode ring overflowed: drain more often (capacity 2*num_games + 64 episodes)");
    return AZ_OK;
}

static int ring_read(az_engine *h, int ring, int64_t ne, int64_t ns, int32_t *ep_slot, int32_t *ep_step, int32_t *ep_len,
                     int64_t *ep_offset, int8_t *ep_outcome, uint64_t *s_bb0, uint64_t *s_bb1, uint8_t *s_player,
                     int32_t *s_counts, cudaStream_t st) {
    const RingPtrs &g = h->rings[ring];
    // destinations may be device memory or pinned host memory
#define CP(dst, src, count, T) if ((dst) && (count) > 0) AZ_CUDA(h, cudaMemcpyAsync((dst), (src), (size_t)(count) * sizeof(T), cudaMemcpyDefault, st))
    CP(ep_slot, g.ep_slot, ne, int32_t); CP(ep_step, g.ep_step, ne, int32_t); CP(ep_len, g.ep_len, ne, int32_t);
    CP(ep_offset, g.ep_offset, ne, int64_t); CP(ep_outcome, g.ep_outcome, ne * 2, int8_t);
    CP(s_bb0, g.s_bb0, ns, uint64_t); CP(s_bb1, g.s_bb1, ns, uint64_t); CP(s_player, g.s_player, ns, uint8_t);
    CP(s_counts, g.s_counts, ns * 7, int32_t);
#undef CP
    return AZ_OK;
}

int32_t az_episode_counts(az_engine *h, int64_t *n_episodes_host, int64_t *n_samples_host, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    return ring_counts(h, h->active_ring, n_episodes_host, n_samples_host, S(stream));
}

int32_t az_drain_episodes(az_engine *h, int64_t ep_cap, int64_t s_cap, int32_t *ep_slot, int32_t *ep_step,
                          int32_t *ep_len, int64_t *ep_offset, int8_t *ep_outcome, uint64_t *s_bb0, uint64_t *s_bb1,
                          uint8_t *s_player, int32_t *s_counts, int64_t *n_episodes_host, int64_t *n_samples_host,
                          void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    int64_t ne = 0, ns = 0;
    cudaStream_t st = S(stream);
    int rc = ring_counts(h, h->active_ring, &ne, &ns, st);
    if (rc != AZ_OK) return rc;
    if (ne > ep_cap || ns > s_cap) return fail(h, AZ_E_OVERFLOW, "%s", "az_drain_episodes: caller buffers too small");
    rc = ring_read(h, h->active_ring, ne, ns, ep_slot, ep_step, ep_len, ep_offset, ep_outcome, s_bb0, s_bb1, s_player, s_counts, st);
    if (rc != AZ_OK) return rc;
    AZ_CUDA(h, cudaMemsetAsync(h->rings[h->active_ring].ring, 0, 4 * sizeof(unsigned long long), st));
    AZ_CUDA(h, cudaStreamSynchronize(st));
    if (n_episodes_host) *n_episodes_host = ne;
    if (n_samples_host) *n_samples_host = ns;
    return AZ_OK;
}

int32_t az_swap_episode_ring(az_engine *h, int32_t *previous_ring_host, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    const int prev = h->active_ring, next = prev ^ 1;
    AZ_CUDA(h, cudaMemsetAsync(h->rings[next].ring, 0, 4 * sizeof(unsigned long long), S(stream)));
    use_ring(h, next);
    if (previous_ring_host) *previous_ring_host = prev;
    return AZ_OK;
}

int32_t az_ring_counts(az_engine *h, int32_t ring, int64_t *n_episodes_host, int64_t *n_samples_host, void *stream) {
    if (!h || ring < 0 || ring > 1) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    return ring_counts(h, ring, n_episodes_host, n_samples_host, S(stream));
}

int32_t az_read_episode_ring(az_engine *h, int32_t ring, int64_t n_episodes, int64_t n_samples, int32_t *ep_slot,
                             int32_t *ep_step, int32_t *ep_len, int64_t *ep_offset, int8_t *ep_outcome, uint64_t *s_bb0,
                             uint64_t *s_bb1, uint8_t *s_player, int32_t *s_counts, void *stream) {
    if (!h || ring < 0 || ring > 1 || n_episodes < 0 || n_samples < 0) return AZ_E_INVALID;
    if (n_episodes > h->a.ep_cap || n_samples > h->a.s_cap) return fail(h, AZ_E_INVALID, "%s", "az_read_episode_ring: counts exceed the ring");
    if (int rc = set_device(h)) return rc;
    return ring_read(h, ring, n_episodes, n_samples, ep_slot, ep_step, ep_len, ep_offset, ep_outcome, s_bb0, s_bb1, s_player, s_counts,
                     S(stream));
}

static int sum_stats(az_engine *h, unsigned long long (&r)[NSTAT], cudaStream_t st) {
    if (int rc = set_device(h)) return rc;
    AZ_CUDA(h, cudaMemsetAsync(h->d_tot, 0, NSTAT * sizeof(unsigned long long), st));
    k_sum_stats<<<148, 256, 0, st>>>(h->a.tstats, h->a.E, h->d_tot);
    AZ_LAUNCH_CHECK(h, "k_sum_stats");
    AZ_CUDA(h, cudaMemcpyAsync(r, h->d_tot, sizeof r, cudaMemcpyDeviceToHost, st));
    AZ_CUDA(h, cudaStreamSynchronize(st));
    for (int q = 0; q < NSTAT; ++q) r[q] += h->acc_tot[q];
    return AZ_OK;
}

int32_t az_get_stats(az_engine *h, az_stats *out, void *stream) {
    if (!h || !out) return AZ_E_INVALID;
    unsigned long long r[NSTAT];
    if (int rc = sum_stats(h, r, S(stream))) return rc;
    out->simulations = r[0];
    out->evaluations = r[1];
    out->levels = r[2];
    out->children_created = r[3];
    out->backup_nodes = r[2] + r[0];
    out->moves = r[4];
    out->episodes = r[5];
    out->children_scanned = r[6];
    return AZ_OK;
}

int32_t az_get_eval_cache_stats(az_engine *h, az_eval_cache_stats *out, void *stream) {
    if (!h || !out) return AZ_E_INVALID;
    unsigned long long r[NSTAT];
    if (int rc = sum_stats(h, r, S(stream))) return rc;
    out->rows = r[1] - r[7] - r[8];
    out->hits = r[7];
    out->followers = r[8];
    out->failed_claims = r[9];
    out->evictions = r[10];
    return AZ_OK;
}

int32_t az_set_eval_cache(az_engine *h, int32_t log2_entries) {
    if (!h) return AZ_E_INVALID;
    if (log2_entries != 0 && (log2_entries < 10 || log2_entries > 30))
        return fail(h, AZ_E_INVALID, "%s", "az_set_eval_cache: log2_entries must be 0 (off) or 10 .. 30");
    if (h->sel_pending && h->cache_sel) return fail(h, AZ_E_STATE, "%s", "az_set_eval_cache: a cached selection waits for its expansion");
    if (log2_entries == h->cache_log2) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    if (h->cache_mem) {
        AZ_CUDA(h, cudaDeviceSynchronize());
        AZ_CUDA(h, cudaFree(h->cache_mem));
        h->bytes -= (int64_t)sizeof(CacheEntry) << h->cache_log2;
        h->cache_mem = nullptr;
    }
    h->a.cache = nullptr;
    h->a.cache_mask = 0;
    h->cache_log2 = 0;
    if (log2_entries == 0) return AZ_OK;
    if (!h->a.leaf_src) {
        const int E = h->a.E;
        int rc = dev_alloc(h, &h->a.leaf_src, E);
        if (rc == AZ_OK) rc = dev_alloc(h, &h->a.leaf_claim, E);
        if (rc == AZ_OK) rc = dev_alloc(h, &h->a.cached_out, (size_t)E * 3);
        if (rc != AZ_OK) return rc;
    }
    const size_t bytes = sizeof(CacheEntry) << log2_entries;
    cudaError_t e = cudaMalloc(&h->cache_mem, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        h->cache_mem = nullptr;
        return fail(h, AZ_E_NOMEM, "az_set_eval_cache: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    AZ_CUDA(h, cudaMemset(h->cache_mem, 0, bytes));  // every entry EMPTY
    h->bytes += (int64_t)bytes;
    h->a.cache = static_cast<CacheEntry *>(h->cache_mem);
    h->a.cache_mask = (1u << (log2_entries - 1)) - 1u;
    h->cache_log2 = log2_entries;
    return AZ_OK;
}

int32_t az_bump_eval_epoch(az_engine *h, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    k_add_u32<<<1, 1, 0, S(stream)>>>(h->a.cache_ctl + 1, 1u);
    AZ_LAUNCH_CHECK(h, "k_add_u32");
    return AZ_OK;
}

int32_t az_selftest_division(az_engine *h, int64_t n, uint64_t seed, int64_t *mismatches_host) {
    if (!h || !mismatches_host || n < 0) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    AZ_CUDA(h, cudaMemset(h->d_tot, 0, 8 * sizeof(unsigned long long)));
    k_selftest_div<<<148 * 8, 256>>>(h->a.rcp, h->a.tab_n - 6, seed, n, h->d_tot);
    AZ_LAUNCH_CHECK(h, "k_selftest_div");
    unsigned long long bad = 0;
    AZ_CUDA(h, cudaMemcpy(&bad, h->d_tot, sizeof bad, cudaMemcpyDeviceToHost));
    *mismatches_host = (int64_t)bad;
    return AZ_OK;
}

int32_t az_reset_stats(az_engine *h, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (int rc = set_device(h)) return rc;
    k_zero_u32<<<148, 256, 0, S(stream)>>>(h->a.tstats, (long long)h->a.E * NSTAT);
    AZ_LAUNCH_CHECK(h, "k_zero_u32");
    memset(h->acc_tot, 0, sizeof h->acc_tot);
    if (h->rstats) AZ_CUDA(h, cudaMemsetAsync(h->rstats, 0, (size_t)h->a.E * RS_N * sizeof(unsigned long long), S(stream)));
    if (h->cap.cstats) AZ_CUDA(h, cudaMemsetAsync(h->cap.cstats, 0, (size_t)h->a.E * CS_N * sizeof(unsigned long long), S(stream)));
    return AZ_OK;
}

int32_t az_set_subtree_reuse(az_engine *h, int32_t max_root_visits) {
    if (!h) return AZ_E_INVALID;
    const int S_ = h->cfg.num_simulations;
    if (max_root_visits != 0 && (max_root_visits < S_ || max_root_visits > AZ_MAX_ROOT_VISITS))
        return fail(h, AZ_E_INVALID, "%s", "az_set_subtree_reuse: max_root_visits must be 0 (off) or in [num_simulations, 65536]");
    if (h->sel_pending) return fail(h, AZ_E_STATE, "%s", "az_set_subtree_reuse: a selection's leaves wait for their expansion");
    if (int rc = set_device(h)) return rc;
    Arena &a = h->a;
    const int E = a.E;
    const int V = max_root_visits ? max_root_visits : S_;
    const int cap = ((1 + 7 * V) + 7) & ~7;
    const int tab_n = V + 8;
    // everything new is allocated before anything old is released: on AZ_E_NOMEM the engine is as it was
    double *W = nullptr;
    uint4 *M = nullptr;
    double *rcp = nullptr, *sqt = nullptr;
    double2 *t2 = nullptr;
    int rc = AZ_OK;
    if (cap != a.cap) {
        rc = dev_alloc(h, &W, (size_t)E * cap);
        if (rc == AZ_OK) rc = dev_alloc(h, &M, (size_t)E * cap);
    }
    if (rc == AZ_OK && tab_n != a.tab_n) {
        rc = dev_alloc(h, &rcp, tab_n);
        if (rc == AZ_OK) rc = dev_alloc(h, &sqt, tab_n);
        if (rc == AZ_OK) rc = dev_alloc(h, &t2, tab_n);
    }
    if (rc == AZ_OK && max_root_visits && !h->reroot) rc = dev_alloc(h, &h->reroot, E);
    if (rc == AZ_OK && max_root_visits && !h->rstats) {
        unsigned long long *p = nullptr;
        rc = dev_alloc(h, &p, (size_t)E * RS_N);
        if (rc == AZ_OK) {
            AZ_CUDA(h, cudaMemset(p, 0, (size_t)E * RS_N * sizeof(unsigned long long)));
            h->rstats = p;
        }
    }
    if (rc != AZ_OK) {
        void *fresh[] = {W, M, rcp, sqt, t2};
        const size_t sz[] = {(size_t)E * cap * sizeof(double), (size_t)E * cap * sizeof(uint4), tab_n * sizeof(double),
                             tab_n * sizeof(double), tab_n * sizeof(double2)};
        for (int i = 0; i < 5; ++i)
            if (fresh[i]) dev_free(h, fresh[i], sz[i]);
        return rc;
    }
    AZ_CUDA(h, cudaDeviceSynchronize());  // no launch may still use what is released below
    if (W) {
        dev_free(h, a.W, (size_t)E * a.cap * sizeof(double));
        dev_free(h, a.M, (size_t)E * a.cap * sizeof(uint4));
        a.W = W;
        a.M = M;
        a.cap = cap;
    }
    if (rcp) {
        dev_free(h, const_cast<double *>(a.rcp), a.tab_n * sizeof(double));
        dev_free(h, const_cast<double *>(a.sqt), a.tab_n * sizeof(double));
        dev_free(h, const_cast<double2 *>(a.t2), a.tab_n * sizeof(double2));
        k_init_tables<<<blocks_for(tab_n, 256), 256>>>(rcp, sqt, t2, tab_n);
        AZ_LAUNCH_CHECK(h, "k_init_tables");
        a.rcp = rcp;
        a.sqt = sqt;
        a.t2 = t2;
        a.tab_n = tab_n;
    }
    k_reset_trees<<<blocks_for(E, 256), 256>>>(a, E);
    AZ_LAUNCH_CHECK(h, "k_reset_trees");
    if (h->cap_on)  // the budgets of the current step count from the reset roots
        if (int rc2 = launch_cap_draw(h, (uint32_t)h->step, false, nullptr)) return rc2;
    AZ_CUDA(h, cudaDeviceSynchronize());
    h->reuse_v = max_root_visits;
    h->sims_done = 0;
    h->noise_applied = false;
    return AZ_OK;
}

int32_t az_advance_roots(az_engine *h, const uint8_t *cols, uint8_t *out_status, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!cols || !out_status) return fail(h, AZ_E_INVALID, "%s", "az_advance_roots: null argument");
    if (h->reuse_v == 0) return fail(h, AZ_E_STATE, "%s", "az_advance_roots: subtree reuse is off (az_set_subtree_reuse)");
    if (h->sel_pending) return fail(h, AZ_E_STATE, "%s", "az_advance_roots: a selection's leaves wait for their expansion");
    if (int rc = set_device(h)) return rc;
    const int n = h->n_active;
    k_advance_roots<<<blocks_for(n, 256), 256, 0, S(stream)>>>(h->a, n, cols, out_status, h->reroot);
    AZ_LAUNCH_CHECK(h, "k_advance_roots");
    if (int rc = launch_reroot(h, n, S(stream))) return rc;
    if (h->cap_on)  // not a self-play move step: every search is full
        if (int rc = launch_cap_draw(h, 0u, true, S(stream))) return rc;
    h->sims_done = 0;
    h->noise_applied = false;
    return AZ_OK;
}

int32_t az_get_reuse_stats(az_engine *h, az_reuse_stats *out, void *stream) {
    if (!h || !out) return AZ_E_INVALID;
    memset(out, 0, sizeof *out);
    if (!h->rstats) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    const size_t n = (size_t)h->a.E * RS_N;
    unsigned long long *buf = (unsigned long long *)malloc(n * sizeof(unsigned long long));
    if (!buf) return fail(h, AZ_E_NOMEM, "%s", "az_get_reuse_stats: host allocation failed");
    cudaError_t e = cudaMemcpyAsync(buf, h->rstats, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, S(stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(S(stream));
    if (e != cudaSuccess) {
        free(buf);
        return fail(h, AZ_E_CUDA, "az_get_reuse_stats: %s", cudaGetErrorString(e));
    }
    unsigned long long tot[RS_N] = {};
    for (size_t i = 0; i < n; ++i) tot[i % RS_N] += buf[i];
    free(buf);
    out->retained = tot[RS_RETAINED];
    out->fresh = tot[RS_FRESH];
    out->dropped = tot[RS_DROPPED];
    out->nodes = tot[RS_NODES];
    out->visits = tot[RS_VISITS];
    return AZ_OK;
}

int32_t az_set_playout_cap(az_engine *h, const az_playout_cap *cfg) {
    if (!h) return AZ_E_INVALID;
    if (h->sel_pending) return fail(h, AZ_E_STATE, "%s", "az_set_playout_cap: a selection's leaves wait for their expansion");
    if (!cfg) {
        h->cap_on = false;
        return AZ_OK;
    }
    const int S_ = h->cfg.num_simulations;
    if (cfg->fast_sims < 1 || cfg->fast_sims > S_)
        return fail(h, AZ_E_INVALID, "%s", "az_set_playout_cap: fast_sims must be in [1, num_simulations]");
    if (!(cfg->p_full >= 0.0f && cfg->p_full <= 1.0f)) return fail(h, AZ_E_INVALID, "%s", "az_set_playout_cap: p_full must be in [0, 1]");
    if (cfg->slot_offset < 0 || cfg->slot_offset > ((int64_t)1 << 62))
        return fail(h, AZ_E_INVALID, "%s", "az_set_playout_cap: slot_offset must be in [0, 2^62]");
    if (cfg->visit_budget != 0 && cfg->visit_budget != 1) return fail(h, AZ_E_INVALID, "%s", "az_set_playout_cap: visit_budget must be 0 or 1");
    if (int rc = set_device(h)) return rc;
    const int E = h->a.E;
    CapArgs &cp = h->cap;
    if (!cp.budget) {
        uint32_t *budget = nullptr;
        uint8_t *full = nullptr, *g_full = nullptr;
        unsigned long long *cstats = nullptr;
        int rc = dev_alloc(h, &budget, E);
        if (rc == AZ_OK) rc = dev_alloc(h, &full, E);
        if (rc == AZ_OK) rc = dev_alloc(h, &g_full, (size_t)E * MAX_PLIES);
        if (rc == AZ_OK) rc = dev_alloc(h, &cstats, (size_t)E * CS_N);
        if (rc != AZ_OK) {
            if (budget) dev_free(h, budget, (size_t)E * sizeof(uint32_t));
            if (full) dev_free(h, full, (size_t)E);
            if (g_full) dev_free(h, g_full, (size_t)E * MAX_PLIES);
            return rc;
        }
        AZ_CUDA(h, cudaMemset(cstats, 0, (size_t)E * CS_N * sizeof(unsigned long long)));
        cp.budget = budget;
        cp.full = full;
        cp.g_full = g_full;
        cp.cstats = cstats;
    }
    // the flags apply only while the mode is on: every ply already in the logs counts as full (az_engine.h)
    if (!h->cap_on) AZ_CUDA(h, cudaMemset(cp.g_full, 1, (size_t)E * MAX_PLIES));
    cp.seed = cfg->seed;
    cp.slot_offset = cfg->slot_offset;
    cp.p_full = (double)cfg->p_full;
    cp.S = S_;
    cp.fast = cfg->fast_sims;
    cp.visit_budget = cfg->visit_budget;
    h->cap_on = true;
    if (int rc = launch_cap_draw(h, (uint32_t)h->step, false, nullptr)) return rc;
    AZ_CUDA(h, cudaDeviceSynchronize());
    return AZ_OK;
}

int32_t az_search_budgets(az_engine *h, uint32_t *budget, uint8_t *full, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (!h->cap.budget) return fail(h, AZ_E_STATE, "%s", "az_search_budgets: no playout cap configured (az_set_playout_cap)");
    if (int rc = set_device(h)) return rc;
    const size_t E = (size_t)h->a.E;
    if (budget) AZ_CUDA(h, cudaMemcpyAsync(budget, h->cap.budget, E * sizeof(uint32_t), cudaMemcpyDefault, S(stream)));
    if (full) AZ_CUDA(h, cudaMemcpyAsync(full, h->cap.full, E, cudaMemcpyDefault, S(stream)));
    return AZ_OK;
}

int32_t az_get_cap_stats(az_engine *h, az_cap_stats *out, void *stream) {
    if (!h || !out) return AZ_E_INVALID;
    memset(out, 0, sizeof *out);
    unsigned long long r[NSTAT];
    if (int rc = sum_stats(h, r, S(stream))) return rc;
    out->simulations = r[0];
    if (!h->cap.cstats) return AZ_OK;
    const size_t n = (size_t)h->a.E * CS_N;
    unsigned long long *buf = (unsigned long long *)malloc(n * sizeof(unsigned long long));
    if (!buf) return fail(h, AZ_E_NOMEM, "%s", "az_get_cap_stats: host allocation failed");
    cudaError_t e = cudaMemcpyAsync(buf, h->cap.cstats, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, S(stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(S(stream));
    if (e != cudaSuccess) {
        free(buf);
        return fail(h, AZ_E_CUDA, "az_get_cap_stats: %s", cudaGetErrorString(e));
    }
    unsigned long long tot[CS_N] = {};
    for (size_t i = 0; i < n; ++i) tot[i % CS_N] += buf[i];
    free(buf);
    out->full_searches = tot[CS_FULL];
    out->fast_searches = tot[CS_FAST];
    out->samples_recorded = tot[CS_RECORDED];
    out->samples_dropped = tot[CS_DROPPED];
    return AZ_OK;
}

int32_t az_set_symmetric_eval(az_engine *h, int32_t on) {
    if (!h) return AZ_E_INVALID;
    if (h->sel_pending) return fail(h, AZ_E_STATE, "%s", "az_set_symmetric_eval: a selection's leaves wait for their expansion");
    if (on && !h->leaf_mirror) {
        if (int rc = set_device(h)) return rc;
        if (int rc = dev_alloc(h, &h->leaf_mirror, h->a.E)) return rc;
        AZ_CUDA(h, cudaMemset(h->leaf_mirror, 0, (size_t)h->a.E));
    }
    h->sym = on != 0;
    return AZ_OK;
}

int32_t az_leaf_mirror(az_engine *h, const uint8_t **mirrored) {
    if (!h || !mirrored) return AZ_E_INVALID;
    *mirrored = h->sym_sel ? h->leaf_mirror : nullptr;
    return AZ_OK;
}

int32_t az_mirror_states(az_engine *h, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *flags, int64_t n, uint64_t *out_bb0,
                         uint64_t *out_bb1, void *stream) {
    if (!h) return AZ_E_INVALID;
    if (n < 0 || (n > 0 && (!bb0 || !bb1 || !out_bb0 || !out_bb1))) return fail(h, AZ_E_INVALID, "%s", "az_mirror_states: null argument");
    if (n == 0) return AZ_OK;
    if (int rc = set_device(h)) return rc;
    const void *ptrs[] = {bb0, bb1, out_bb0, out_bb1};
    bool vec = !flags || (reinterpret_cast<uintptr_t>(flags) & 3u) == 0;
    for (const void *p : ptrs) vec = vec && (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
    const long long quads = vec ? n / 4 : 0, head = quads * 4;
    if (quads) {
        k_mirror_states<<<blocks_for(quads, 256), 256, 0, S(stream)>>>(bb0, bb1, flags, n, out_bb0, out_bb1, 1);
        AZ_LAUNCH_CHECK(h, "k_mirror_states");
    }
    if (head < n) {
        k_mirror_states<<<blocks_for(n - head, 256), 256, 0, S(stream)>>>(bb0 + head, bb1 + head, flags ? flags + head : nullptr, n - head,
                                                                      out_bb0 + head, out_bb1 + head, 0);
        AZ_LAUNCH_CHECK(h, "k_mirror_states");
    }
    return AZ_OK;
}

}  // extern "C"
