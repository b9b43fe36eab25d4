/*
 * TEST INFRASTRUCTURE — the library's opt-in opening positions (az_set_openings) restated on top of the forced-playouts oracle
 * (tests/native/c4_forced_oracle.c, which includes the cap, reuse and noise oracles and oracle/c4_oracle.c; all included unchanged).
 * The reference has no such option, so there are no goldens: tests/test_oracle_openings.py pins opening_of() to a plain-Python
 * restatement and c4o_selfplay_openings to c4o_selfplay_forced with the mode off.
 *
 * Only what the mode adds is written here (the rule is the one in include/az_engine.h):
 *   - opening_of(): the opening of the game of global slot g that starts at move step s - Philox4x32-10 (the cap oracle's) keyed by
 *     the seed with counter {g lo, g hi, s, 0xA0000000 | j}; the base (entry (X_0.x * n) >> 32 of the set, or the initial state);
 *     r = min + ((X_0.y * (max - min + 1)) >> 32) plies, each among the columns whose drop (play_into, on cells) neither wins nor
 *     fills the board, ascending, candidate (X_j.x * count) >> 32; an ended base or no candidate left stops the plies;
 *   - c4o_openings: opening_of() over n consecutive global slots;
 *   - c4o_selfplay_openings: the c4o_selfplay_forced loop (same arguments and outputs, plus the configuration; NULL = off) in which
 *     every slot starts its first game from opening_of(g, 0) and a slot recycled at move step t from opening_of(g, t + 1).
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (tests/openings_oracle.py, into a temporary directory).
 */
#include "c4_forced_oracle.c"

typedef struct {
    const uint64_t *bb0, *bb1;
    const uint8_t *player;
    int32_t n_positions, min_plies, max_plies;
    uint64_t seed;
    int64_t slot_offset;
} c4o_openings_cfg;

static void open_draw(const c4o_openings_cfg *op, uint64_t g, uint32_t s, uint32_t j, uint32_t x[4]) {
    x[0] = (uint32_t)g; x[1] = (uint32_t)(g >> 32); x[2] = s; x[3] = 0xA0000000u | j;
    philox4x32_10(x, (uint32_t)op->seed, (uint32_t)(op->seed >> 32));
}

/* the opening of the game (g, s) as a fresh root node; (b0, b1, pl) = the base when the set is empty */
static void opening_of(const c4o_openings_cfg *op, uint64_t g, uint32_t s, uint64_t b0, uint64_t b1, int pl, node_t *out) {
    uint32_t x0[4];
    open_draw(op, g, s, 0u, x0);
    if (op->n_positions > 0) {
        const int i = (int)(((uint64_t)x0[0] * (uint64_t)op->n_positions) >> 32);
        b0 = op->bb0[i]; b1 = op->bb1[i]; pl = op->player[i];
    }
    const int r = op->min_plies + (int)(((uint64_t)x0[1] * (uint64_t)(op->max_plies - op->min_plies + 1)) >> 32);
    node_t cur, nx;
    init_root(&cur, b0, b1, pl);
    for (int j = 1; j <= r && !cur.ended; j++) {
        int cand[7], k = 0;
        for (int c = 0; c < 7; c++)
            if (play_into(&cur, c, &nx) == 0 && !nx.ended) cand[k++] = c;
        if (k == 0) break;
        uint32_t x[4];
        open_draw(op, g, s, (uint32_t)j, x);
        play_into(&cur, cand[((uint64_t)x[0] * (uint64_t)k) >> 32], &nx);
        memcpy(cur.cell, nx.cell, NCELL);
        cur.player = nx.player;
    }
    bb_from_cells(cur.cell, &b0, &b1);
    init_root(out, b0, b1, cur.player);
}

/* openings of global slots g0 .. g0 + n - 1 at move step s */
void c4o_openings(const c4o_openings_cfg *op, int64_t g0, int n, uint32_t s, uint64_t init0, uint64_t init1, int initpl, uint64_t *o0,
                  uint64_t *o1, uint8_t *opl) {
    for (int i = 0; i < n; i++) {
        node_t r;
        opening_of(op, (uint64_t)(g0 + i), s, init0, init1, initpl, &r);
        bb_from_cells(r.cell, &o0[i], &o1[i]);
        opl[i] = r.player;
    }
}

/* the root of the game slot i starts at move step s: its opening, or the initial state with the mode off */
static void start_game(const c4o_openings_cfg *op, const c4o_selfplay_cfg *cfg, int i, uint32_t s, node_t *root) {
    if (op) opening_of(op, (uint64_t)(op->slot_offset + i), s, cfg->init_bb0, cfg->init_bb1, cfg->init_player, root);
    else init_root(root, cfg->init_bb0, cfg->init_bb1, cfg->init_player);
}

/* c4o_selfplay_forced (same arguments and outputs) with the games starting from their openings (op NULL = off) */
int c4o_selfplay_openings(const c4o_selfplay_cfg *cfg, const c4o_openings_cfg *op, double k, int V, int fast_sims, int visit_budget, const uint8_t *full,
                        const double *uniforms, c4o_eval_cb cb, void *user, float eps, const float *eta, int greedy_from, int32_t *ep_slot,
                        int32_t *ep_len, int32_t *ep_step, int8_t *ep_outcome, uint64_t *s_bb0, uint64_t *s_bb1, uint8_t *s_player,
                        int32_t *s_counts, int64_t max_samples, int64_t *n_episodes_out, int64_t *n_samples_out, int64_t *n_steps_out,
                        int64_t *n_uniforms_used, int64_t *n_sims_out, int64_t *n_evals_out, int64_t *n_dropped_out, int64_t *st,
                        int64_t *fst, int32_t *last_counts) {
    int E = cfg->E, S = cfg->S;
    if ((V && V < S) || fast_sims < 1 || fast_sims > S) return 1;
    tree_t *trees = alloc_trees(E, V ? V : S);
    tree_t *live = calloc(E > 0 ? (size_t)E : 1, sizeof *live);
    uint8_t *live_full = calloc(E > 0 ? (size_t)E : 1, 1);
    int32_t *n = calloc(E > 0 ? (size_t)E : 1, sizeof *n);
    if (!trees || !live || !live_full || !n) return 1;
    uint64_t *h_bb0 = malloc(8 * (size_t)E * 42), *h_bb1 = malloc(8 * (size_t)E * 42);
    uint8_t *h_pl = malloc((size_t)E * 42), *h_full = malloc((size_t)E * 42);
    int32_t *h_cnt = malloc(sizeof(int32_t) * (size_t)E * 42 * 7);
    int *h_len = calloc((size_t)E, sizeof(int));
    int64_t n_ep = 0, n_s = 0, n_u = 0, n_sims = 0, n_ev = 0, n_drop = 0;
    int err = 0, step = 0, done = 0;
    for (int q = 0; q < RO_N; q++) st[q] = 0;
    for (int q = 0; q < FO_N; q++) fst[q] = 0;
    for (int i = 0; i < E; i++) {
        start_game(op, cfg, i, 0u, &trees[i].nodes[0]);
        trees[i].used = 1;
    }
    while (!done && !err) {
        if (step >= cfg->max_steps) break;
        const uint8_t *fl = &full[(size_t)step * E];
        for (int i = 0; i < E; i++) {
            const int st_i = fl[i] ? S : fast_sims, n0 = trees[i].nodes[0].N;
            n[i] = !visit_budget ? st_i : (st_i > n0 + 1 ? st_i - n0 : 1);
            n_sims += n[i];
        }
        err = run_budgeted_forced(trees, E, n, cfg->c_puct, cfg->eval_kind, cb, user, &n_ev, eps, eta ? &eta[(size_t)step * E * 7] : NULL,
                                  fl, live, live_full, k, &fst[FO_SELECTIONS]);
        if (err) break;
        if (V) note_used(trees, E, st);
        for (int i = 0; i < E; i++) {
            tree_t *t = &trees[i];
            node_t *r = &t->nodes[0];
            int l = h_len[i];
            if (l >= 42) { err = 6; break; }
            size_t o = (size_t)i * 42 + l;
            bb_from_cells(r->cell, &h_bb0[o], &h_bb1[o]);
            h_pl[o] = r->player;
            h_full[o] = fl[i];
            int32_t raw[7] = {0};
            double W[7] = {0};
            float P[7] = {0};
            for (int j = 0; j < r->nchild; j++) {
                node_t *ch = &t->nodes[r->first_child + j];
                raw[ch->col] = ch->N; W[ch->col] = ch->W; P[ch->col] = (float)ch->P;
            }
            const uint8_t legal = legal_mask_of(r);
            if (fl[i]) {
                prune(raw, W, P, legal, r->N, cfg->c_puct, k, &h_cnt[o * 7], &fst[FO_PRUNED], &fst[FO_ZEROED]);
                fst[FO_SEARCHES]++;
            } else {
                memcpy(&h_cnt[o * 7], raw, sizeof raw);
            }
            h_len[i] = l + 1;
            if (last_counts && step == cfg->max_steps - 1) memcpy(&last_counts[(size_t)7 * i], &h_cnt[o * 7], sizeof(int32_t) * 7);
            const double u = uniforms[(size_t)step * E + i];
            int j = (greedy_from >= 0 && l >= greedy_from) ? greedy_child(t) : fl[i] ? sample_counts(&h_cnt[o * 7], legal, u) : sample_child(t, u);
            n_u++;
            node_t next = t->nodes[r->first_child + j];
            if (!next.ended) {
                if (V) {
                    err = keep_subtree(t, r->first_child + j, S, V, st);
                    if (err) break;
                } else {
                    fresh_root(t, &next);
                }
                continue;
            }
            int rec = 0;
            for (int q = 0; q < h_len[i]; q++) rec += h_full[(size_t)i * 42 + q] != 0;
            if (n_s + rec > max_samples) { err = 7; break; }
            ep_slot[n_ep] = i; ep_len[n_ep] = rec; ep_step[n_ep] = step;
            ep_outcome[2 * n_ep] = next.reward0; ep_outcome[2 * n_ep + 1] = (int8_t)-next.reward0;
            for (int q = 0; q < h_len[i]; q++) {
                size_t p = (size_t)i * 42 + q;
                if (!h_full[p]) continue;
                s_bb0[n_s] = h_bb0[p]; s_bb1[n_s] = h_bb1[p]; s_player[n_s] = h_pl[p];
                memcpy(&s_counts[n_s * 7], &h_cnt[p * 7], sizeof(int32_t) * 7);
                n_s++;
            }
            n_drop += h_len[i] - rec;
            n_ep++;
            h_len[i] = 0;
            start_game(op, cfg, i, (uint32_t)step + 1u, &t->nodes[0]);
            t->used = 1;
            if (n_ep >= cfg->quota) { done = 1; break; }
        }
        step++;
    }
    *n_episodes_out = n_ep; *n_samples_out = n_s; *n_steps_out = step; *n_uniforms_used = n_u;
    *n_sims_out = n_sims; *n_evals_out = n_ev; *n_dropped_out = n_drop;
    free(h_bb0); free(h_bb1); free(h_pl); free(h_full); free(h_cnt); free(h_len); free(n); free(live); free(live_full);
    free_trees(trees, E);
    return err;
}
