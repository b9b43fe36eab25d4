/*
 * TEST INFRASTRUCTURE — the library's opt-in playout cap randomization (az_set_playout_cap, KataGo's "playout cap randomization")
 * restated on top of the reuse oracle (tests/native/c4_reuse_oracle.c, which includes the noise oracle and oracle/c4_oracle.c;
 * all included unchanged).  The reference has no such option, so there are no goldens: tests/test_oracle_playout_cap.py pins this
 * file to c4o_selfplay / c4o_selfplay_noise (every search full) and to the same games with every sample dropped.
 *
 * Only what the cap adds is written here:
 *   - per-tree budgets: the search of slot i at move step k runs n = S (full) or fast_sims (fast) new simulations; with
 *     visit_budget n = max(S_t - N_start, 1), N_start = the root's visits at the start of the search (non-zero only with reuse);
 *     the trees run in lockstep, one simulation at a time over the trees that still have simulations to run;
 *   - root noise only on full trees, after the first simulation of the step;
 *   - every move is played and logged, but a finished game emits only the samples of its full searches (ep_len = their number,
 *     possibly 0);
 *   - c4o_cap_draw: the engine's full / fast draw (Philox4x32-10 keyed by the seed, counter {global slot lo, hi, step, 0xC0000000},
 *     full iff (x + 0.5) / 2^32 < p_full), for the test that pins the numpy restatement.
 * The full flags are supplied by the caller (the GPU tests read back what the engine drew), as eta is for the noise oracle.
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (tests/cap_oracle.py, into a temporary directory).
 */
#include "c4_reuse_oracle.c"

static void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

/* full[i] of global slots slot_offset + i, i < n, at move step `step` */
void c4o_cap_draw(uint64_t seed, int64_t slot_offset, int n, uint32_t step, float p_full, uint8_t *full) {
    for (int i = 0; i < n; i++) {
        const uint64_t g = (uint64_t)(slot_offset + i);
        uint32_t c[4] = {(uint32_t)g, (uint32_t)(g >> 32), step, 0xC0000000u};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        full[i] = (((double)c[0] + 0.5) * 0x1p-32) < (double)p_full;
    }
}

/* simulations of every tree up to its budget n[i], in lockstep; eta: the noise on the full trees after the first simulation */
static int run_budgeted(tree_t *trees, int E, const int32_t *n, double c_puct, int kind, c4o_eval_cb cb, void *user, int64_t *n_evals,
                        float eps, const float *eta, const uint8_t *full, tree_t *live) {
    int maxn = 0;
    for (int i = 0; i < E; i++) maxn = n[i] > maxn ? n[i] : maxn;
    for (int s = 0; s < maxn; s++) {
        if (s == 1 && eta)
            for (int i = 0; i < E; i++)
                if (full[i] && trees[i].nodes[0].nchild > 0) mix_root_noise(&trees[i], eps, &eta[(size_t)7 * i]);
        int m = 0;
        for (int i = 0; i < E; i++) if (s < n[i]) live[m++] = trees[i];
        const int err = run_sims(live, m, 1, c_puct, kind, cb, user, n_evals);
        for (int i = 0, j = 0; i < E; i++) if (s < n[i]) trees[i] = live[j++];
        if (err) return err;
    }
    return 0;
}

/* c4o_selfplay_reuse (same loop; V = 0: no reuse, the played child becomes a fresh root) with the playout cap: full[step][E] the
 * engine's flags, fast_sims, visit_budget.  ep_len / the samples hold the full searches only; n_sims_out = the new simulations
 * run; n_dropped_out = samples of finished games left out.  st[RO_N] the reuse counters.  last_counts [E][7] (or NULL): the root
 * visit counts by column that the last move step's search left, recorded whether or not its game ended. */
int c4o_selfplay_cap(const c4o_selfplay_cfg *cfg, int V, int fast_sims, int visit_budget, const uint8_t *full, const double *uniforms,
                     c4o_eval_cb cb, void *user, float eps, const float *eta, int greedy_from, int32_t *ep_slot, int32_t *ep_len,
                     int32_t *ep_step, int8_t *ep_outcome, uint64_t *s_bb0, uint64_t *s_bb1, uint8_t *s_player, int32_t *s_counts,
                     int64_t max_samples, int64_t *n_episodes_out, int64_t *n_samples_out, int64_t *n_steps_out,
                     int64_t *n_uniforms_used, int64_t *n_sims_out, int64_t *n_evals_out, int64_t *n_dropped_out, int64_t *st,
                     int32_t *last_counts) {
    int E = cfg->E, S = cfg->S;
    if ((V && V < S) || fast_sims < 1 || fast_sims > S) return 1;
    tree_t *trees = alloc_trees(E, V ? V : S);
    tree_t *live = calloc(E > 0 ? (size_t)E : 1, sizeof *live);
    int32_t *n = calloc(E > 0 ? (size_t)E : 1, sizeof *n);
    if (!trees || !live || !n) return 1;
    uint64_t *h_bb0 = malloc(8 * (size_t)E * 42), *h_bb1 = malloc(8 * (size_t)E * 42);
    uint8_t *h_pl = malloc((size_t)E * 42), *h_full = malloc((size_t)E * 42);
    int32_t *h_cnt = malloc(sizeof(int32_t) * (size_t)E * 42 * 7);
    int *h_len = calloc((size_t)E, sizeof(int));
    int64_t n_ep = 0, n_s = 0, n_u = 0, n_sims = 0, n_ev = 0, n_drop = 0;
    int err = 0, step = 0, done = 0;
    for (int k = 0; k < RO_N; k++) st[k] = 0;
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
        err = run_budgeted(trees, E, n, cfg->c_puct, cfg->eval_kind, cb, user, &n_ev, eps, eta ? &eta[(size_t)step * E * 7] : NULL, fl, live);
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
            for (int c = 0; c < 7; c++) h_cnt[o * 7 + c] = 0;
            for (int j = 0; j < r->nchild; j++) {
                node_t *ch = &t->nodes[r->first_child + j];
                h_cnt[o * 7 + ch->col] = ch->N;
            }
            h_len[i] = l + 1;
            if (last_counts && step == cfg->max_steps - 1) memcpy(&last_counts[(size_t)7 * i], &h_cnt[o * 7], sizeof(int32_t) * 7);
            const double u = uniforms[(size_t)step * E + i];
            int j = (greedy_from >= 0 && l >= greedy_from) ? greedy_child(t) : sample_child(t, u);
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
            for (int k = 0; k < h_len[i]; k++) rec += h_full[(size_t)i * 42 + k] != 0;
            if (n_s + rec > max_samples) { err = 7; break; }
            ep_slot[n_ep] = i; ep_len[n_ep] = rec; ep_step[n_ep] = step;
            ep_outcome[2 * n_ep] = next.reward0; ep_outcome[2 * n_ep + 1] = (int8_t)-next.reward0;
            for (int k = 0; k < h_len[i]; k++) {
                size_t q = (size_t)i * 42 + k;
                if (!h_full[q]) continue;
                s_bb0[n_s] = h_bb0[q]; s_bb1[n_s] = h_bb1[q]; s_player[n_s] = h_pl[q];
                memcpy(&s_counts[n_s * 7], &h_cnt[q * 7], sizeof(int32_t) * 7);
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
    free(h_bb0); free(h_bb1); free(h_pl); free(h_full); free(h_cnt); free(h_len); free(n); free(live);
    free_trees(trees, E);
    return err;
}
