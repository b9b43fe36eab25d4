/*
 * TEST INFRASTRUCTURE — the library's opt-in forced playouts and policy target pruning (az_set_forced_playouts, KataGo, Wu 2019
 * section 3.1) restated on top of the cap oracle (tests/native/c4_cap_oracle.c, which includes the reuse and noise oracles and
 * oracle/c4_oracle.c; all included unchanged).  The reference has no such option, so there are no goldens:
 * tests/test_oracle_forced_playouts.py pins this file to c4o_selfplay_cap / c4o_selfplay_noise / c4o_selfplay at k = 0 and to a
 * numpy restatement of the pruning.
 *
 * Only what the mode adds is written here (the rule is the one in include/az_engine.h; every fp64 operation rounds on its own):
 *   - descend_forced(): at the root, with m = N_root - 1, the first child (ascending column) with N * N < (k * P) * m is taken
 *     before any PUCT score; below the root select_child() as before.  oracle/c4_oracle.c's descend() is static and fixed, so
 *     run_sims() is copied here with descend_forced() in it (built-in and callback paths);
 *   - prune(): the pruned counts N' of one root, one playout at a time;
 *   - c4o_selfplay_forced: the c4o_selfplay_cap loop with forcing on the full trees (every tree without the cap: full all 1), the
 *     pruned counts as the samples of those searches and the move drawn from them (p = N' / sum N' through the same
 *     cumsum / normalise / searchsorted-right), and the mode's counters.
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (tests/forced_oracle.py, into a temporary directory).
 */
#include "c4_cap_oracle.c"

enum { FO_SELECTIONS, FO_SEARCHES, FO_PRUNED, FO_ZEROED, FO_N };

/* descend() with the forced rule at the root of a forced tree; *forced += 1 when the rule decided the root selection */
static int descend_forced(const tree_t *t, double c_puct, double k, int force, int64_t *forced) {
    int ni = 0;
    const node_t *r = &t->nodes[0];
    if (force && r->nchild > 0) {
        const double m = (double)(r->N - 1);
        for (int i = 0; i < r->nchild; i++) {
            const node_t *ch = &t->nodes[r->first_child + i];
            if ((double)ch->N * (double)ch->N < (k * ch->P) * m) {
                ni = r->first_child + i;
                (*forced)++;
                break;
            }
        }
    }
    while (t->nodes[ni].nchild > 0) ni = select_child(t, ni, c_puct);
    return ni;
}

/* simulate_builtin() with descend_forced() */
static int simulate_builtin_forced(tree_t *t, double c_puct, int kind, double k, int force, int64_t *forced, int *err) {
    int leaf = descend_forced(t, c_puct, k, force, forced);
    node_t *n = &t->nodes[leaf];
    if (n->ended) {
        if (n->parent < 0) { *err = 3; return 0; }
        backprop(t, leaf, reward_of(n, t->nodes[n->parent].player));
        return 0;
    }
    float pri[7], val[2];
    uint8_t legal = legal_mask_of(n);
    builtin_eval(kind, n, legal, pri, val);
    if (expand(t, leaf, legal, pri)) { *err = 4; return 0; }
    backprop(t, leaf, (double)val[n->player]);
    return 1;
}

/* run_sims() with descend_forced(): tree i is forced when force[i] */
static int run_sims_forced(tree_t *trees, int E, int S, double c_puct, int kind, c4o_eval_cb cb, void *user, int64_t *n_evals,
                           double k, const uint8_t *force, int64_t *forced) {
    int err = 0;
    int64_t evals = 0, nf = 0;
    if (!cb) {
#pragma omp parallel for schedule(dynamic, 8) reduction(+ : evals, nf) reduction(| : err)
        for (int i = 0; i < E; i++) {
            int e = 0;
            for (int s = 0; s < S; s++) evals += simulate_builtin_forced(&trees[i], c_puct, kind, k, force[i], &nf, &e);
            err |= e;
        }
        if (n_evals) *n_evals += evals;
        *forced += nf;
        return err;
    }
    int *leaf = malloc(sizeof(int) * E), *slot = malloc(sizeof(int) * E), *sel = malloc(sizeof(int) * E);
    uint64_t *b0 = malloc(8 * E), *b1 = malloc(8 * E);
    uint8_t *pl = malloc(E), *lg = malloc(E);
    float *pri = malloc(sizeof(float) * 7 * E), *val = malloc(sizeof(float) * 2 * E);
    for (int s = 0; s < S && !err; s++) {
#pragma omp parallel for schedule(static) reduction(+ : nf) reduction(| : err)
        for (int i = 0; i < E; i++) {
            tree_t *t = &trees[i];
            int l = descend_forced(t, c_puct, k, force[i], &nf);
            node_t *n = &t->nodes[l];
            sel[i] = -1;
            if (n->ended) {
                if (n->parent < 0) { err |= 3; continue; }
                backprop(t, l, reward_of(n, t->nodes[n->parent].player));
            } else {
                sel[i] = l;
            }
        }
        if (err) break;
        int nb = 0;
        for (int i = 0; i < E; i++) {
            if (sel[i] < 0) continue;
            node_t *n = &trees[i].nodes[sel[i]];
            leaf[nb] = sel[i]; slot[nb] = i;
            bb_from_cells(n->cell, &b0[nb], &b1[nb]);
            pl[nb] = n->player; lg[nb] = legal_mask_of(n);
            nb++;
        }
        if (nb == 0) continue;
        cb(user, nb, b0, b1, pl, lg, pri, val);
        evals += nb;
#pragma omp parallel for schedule(static) reduction(| : err)
        for (int j = 0; j < nb; j++) {
            tree_t *t = &trees[slot[j]];
            if (expand(t, leaf[j], lg[j], &pri[7 * j])) { err |= 4; continue; }
            backprop(t, leaf[j], (double)val[2 * j + pl[j]]);
        }
    }
    free(leaf); free(slot); free(sel); free(b0); free(b1); free(pl); free(lg); free(pri); free(val);
    if (n_evals) *n_evals += evals;
    *forced += nf;
    return err;
}

/* run_budgeted() with forcing on the full trees */
static int run_budgeted_forced(tree_t *trees, int E, const int32_t *n, double c_puct, int kind, c4o_eval_cb cb, void *user,
                               int64_t *n_evals, float eps, const float *eta, const uint8_t *full, tree_t *live, uint8_t *live_full,
                               double k, int64_t *forced) {
    int maxn = 0;
    for (int i = 0; i < E; i++) maxn = n[i] > maxn ? n[i] : maxn;
    for (int s = 0; s < maxn; s++) {
        if (s == 1 && eta)
            for (int i = 0; i < E; i++)
                if (full[i] && trees[i].nodes[0].nchild > 0) mix_root_noise(&trees[i], eps, &eta[(size_t)7 * i]);
        int m = 0;
        for (int i = 0; i < E; i++)
            if (s < n[i]) { live_full[m] = full[i]; live[m++] = trees[i]; }
        const int err = run_sims_forced(live, m, 1, c_puct, kind, cb, user, n_evals, k, live_full, forced);
        for (int i = 0, j = 0; i < E; i++) if (s < n[i]) trees[i] = live[j++];
        if (err) return err;
    }
    return 0;
}

/* The pruned counts of one root: cnt / W / P by column (0 off `legal`), root_n = N_root.  *pruned += sum N - N',
 * *zeroed += children that went from N > 0 to 0. */
static void prune(const int32_t *cnt, const double *W, const float *P, uint8_t legal, int32_t root_n, double c_puct, double k,
                  int32_t *out, int64_t *pruned, int64_t *zeroed) {
    for (int c = 0; c < 7; c++) out[c] = cnt[c];
    if (root_n <= 1 || k == 0.0) return;
    const double m = (double)(root_n - 1);
    int bc = -1;
    for (int c = 0; c < 7; c++)
        if ((legal >> c & 1) && (bc < 0 || cnt[c] > cnt[bc])) bc = c;
    const double sq = sqrt((double)root_n);
    const double q_star = W[bc] == 0.0 ? 0.0 : W[bc] / (double)cnt[bc];
    const double s_star = q_star + ((c_puct * (double)P[bc]) * sq) / (double)(1 + cnt[bc]);
    for (int c = 0; c < 7; c++) {
        if (!(legal >> c & 1) || c == bc || cnt[c] <= 0) continue;
        const int32_t n = cnt[c];
        const double q = W[c] == 0.0 ? 0.0 : W[c] / (double)n;
        const double x = (c_puct * (double)P[c]) * sq;
        const double thr = (k * (double)P[c]) * m;
        int32_t nf = 0;
        while ((double)nf * (double)nf < thr) nf++;
        int32_t np = n;
        while (n - np < nf && np > 0 && q + x / (double)np < s_star) np--; /* u(N' - 1) = x / (1 + N' - 1) */
        if (np == 1) np = 0;
        *pruned += n - np;
        *zeroed += np == 0;
        out[c] = np;
    }
}

/* n roots: N / W / P [n][7] by column, legal [n], root_N [n] -> out [n][7]; st[2] = visits pruned, children zeroed */
void c4o_prune(int n, const int32_t *N, const double *W, const float *P, const uint8_t *legal, const int32_t *root_N, double c_puct,
               double k, int32_t *out, int64_t *st) {
    st[0] = st[1] = 0;
    for (int i = 0; i < n; i++)
        prune(&N[(size_t)7 * i], &W[(size_t)7 * i], &P[(size_t)7 * i], legal[i], root_N[i], c_puct, k, &out[(size_t)7 * i], &st[0], &st[1]);
}

/* select_next_node on counts by column: p = cnt / sum cnt over the legal columns; returns the child index (insertion order) */
static int sample_counts(const int32_t *cnt, uint8_t legal, double u) {
    double cdf[MAXCH];
    int32_t sum = 0;
    for (int c = 0; c < 7; c++) if (legal >> c & 1) sum += cnt[c];
    const double denom = (double)sum;
    double acc = 0.0;
    int k = 0;
    for (int c = 0; c < 7; c++) {
        if (!(legal >> c & 1)) continue;
        const double p = (double)cnt[c] / denom;
        acc = (k == 0) ? p : acc + p;
        cdf[k++] = acc;
    }
    const double last = cdf[k - 1];
    int idx = 0;
    for (int i = 0; i < k; i++) cdf[i] /= last;
    while (idx < k && cdf[idx] <= u) idx++;
    if (idx >= k) idx = k - 1;
    return idx;
}

/* c4o_selfplay_cap (same arguments, same outputs) with forced playouts of parameter k on the full searches: their samples are
 * the pruned counts and their moves are drawn from them.  fst[FO_N]: root selections the rule decided, forced searches that
 * ended in a move, visits pruned, children pruned to 0.  last_counts: the recorded (pruned) counts of the last move step. */
int c4o_selfplay_forced(const c4o_selfplay_cfg *cfg, double k, int V, int fast_sims, int visit_budget, const uint8_t *full,
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
        init_root(&trees[i].nodes[0], cfg->init_bb0, cfg->init_bb1, cfg->init_player);
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
            init_root(&t->nodes[0], cfg->init_bb0, cfg->init_bb1, cfg->init_player);
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
