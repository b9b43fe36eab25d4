/*
 * TEST INFRASTRUCTURE — the library's opt-in self-play exploration restated on top of the C oracle: root noise
 * (add_exploration_noise of deepmind_alphazero_pseudocode.py, as az_apply_root_noise does it) and the greedy cutoff
 * (select_action past num_sampling_moves, as az_set_greedy_from does it).  The reference ships both as pseudocode only and
 * never calls them, so there are no goldens: tests/test_oracle_root_noise.py pins this file to c4o_selfplay (noise off), to the
 * numpy fp32 formula and to the first-argmax rule.
 *
 * The search, the rules, the evaluators and the sampling are oracle/c4_oracle.c itself, included unchanged as part of this
 * translation unit.  Only what the noise adds is written here:
 *   - a search runs simulation 1, then every expanded root child's prior becomes RN(RN(RN(1 - eps) * P) + RN(eps * eta[col]))
 *     in fp32 with one rounding per operation (-ffp-contract=off), then simulations 2 .. S;
 *   - from ply greedy_from of a game on, the move is the most visited root child, the first one on ties; the uniform of the
 *     slot is consumed all the same.
 * eta is supplied by the caller (the GPU tests read back what the engine drew): this checks the search around the noise,
 * not the sampler.
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (tests/noise_oracle.py, into a temporary directory).
 */
#include "../../oracle/c4_oracle.c"

static void mix_root_noise(tree_t *t, float eps, const float *eta /*[7]*/) {
    node_t *r = &t->nodes[0];
    const float keep = 1.0f - eps;
    for (int j = 0; j < r->nchild; j++) {
        node_t *ch = &t->nodes[r->first_child + j];
        const float a = keep * (float)ch->P;
        const float b = eps * eta[ch->col];
        const float p = a + b;
        ch->P = (double)p;
    }
}

/* S simulations; with eta != NULL: one simulation, the noise on every expanded root, the other S - 1 */
static int run_sims_noise(tree_t *trees, int E, int S, double c_puct, int kind, c4o_eval_cb cb, void *user, int64_t *n_evals,
                          float eps, const float *eta /*[E][7] or NULL*/) {
    if (!eta || S < 1) return run_sims(trees, E, S, c_puct, kind, cb, user, n_evals);
    int err = run_sims(trees, E, 1, c_puct, kind, cb, user, n_evals);
    if (err) return err;
    for (int i = 0; i < E; i++)
        if (trees[i].nodes[0].nchild > 0) mix_root_noise(&trees[i], eps, &eta[(size_t)7 * i]);
    return run_sims(trees, E, S - 1, c_puct, kind, cb, user, n_evals);
}

/* the most visited root child, the first one on ties (insertion order = ascending column) */
static int greedy_child(const tree_t *t) {
    const node_t *r = &t->nodes[0];
    int best = 0;
    for (int i = 1; i < r->nchild; i++)
        if (t->nodes[r->first_child + i].N > t->nodes[r->first_child + best].N) best = i;
    return best;
}

/* c4o_search with the noise (eps, eta[E][7]) between simulation 1 and simulation 2; child_P = the mixed priors */
int c4o_search_noise(int E, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int S, double c_puct,
                     int eval_kind, c4o_eval_cb cb, void *user, float eps, const float *eta, int32_t *child_N, double *child_W,
                     float *child_P, double *root_W, int32_t *root_N, uint8_t *legal_out, int64_t *n_evals) {
    tree_t *trees = alloc_trees(E, S);
    if (!trees) return 1;
    for (int i = 0; i < E; i++) { init_root(&trees[i].nodes[0], bb0[i], bb1[i], player[i]); trees[i].used = 1; }
    int64_t ev = 0;
    int err = run_sims_noise(trees, E, S, c_puct, eval_kind, cb, user, &ev, eps, eta);
    for (int i = 0; i < E; i++) {
        node_t *r = &trees[i].nodes[0];
        for (int c = 0; c < 7; c++) { child_N[7 * i + c] = 0; child_W[7 * i + c] = 0.0; child_P[7 * i + c] = 0.0f; }
        for (int j = 0; j < r->nchild; j++) {
            node_t *ch = &trees[i].nodes[r->first_child + j];
            child_N[7 * i + ch->col] = ch->N; child_W[7 * i + ch->col] = ch->W; child_P[7 * i + ch->col] = (float)ch->P;
        }
        root_W[i] = r->W; root_N[i] = r->N; legal_out[i] = legal_mask_of(r);
    }
    if (n_evals) *n_evals = ev;
    free_trees(trees, E);
    return err;
}

/* c4o_selfplay (same loop, same outputs) with the noise of every move step's search (eps; eta[step][E][7]) and the greedy
 * cutoff (plies >= greedy_from play greedy_child; negative = off) */
int c4o_selfplay_noise(const c4o_selfplay_cfg *cfg, const double *uniforms, c4o_eval_cb cb, void *user, float eps,
                       const float *eta, int greedy_from, int32_t *ep_slot, int32_t *ep_len, int32_t *ep_step,
                       int8_t *ep_outcome, uint64_t *s_bb0, uint64_t *s_bb1, uint8_t *s_player, int32_t *s_counts,
                       int64_t max_samples, int64_t *n_episodes_out, int64_t *n_samples_out, int64_t *n_steps_out,
                       int64_t *n_uniforms_used, int64_t *n_sims_out, int64_t *n_evals_out) {
    int E = cfg->E, S = cfg->S;
    tree_t *trees = alloc_trees(E, S);
    if (!trees) return 1;
    uint64_t *h_bb0 = malloc(8 * (size_t)E * 42), *h_bb1 = malloc(8 * (size_t)E * 42);
    uint8_t *h_pl = malloc((size_t)E * 42);
    int32_t *h_cnt = malloc(sizeof(int32_t) * (size_t)E * 42 * 7);
    int *h_len = calloc((size_t)E, sizeof(int));
    int64_t n_ep = 0, n_s = 0, n_u = 0, n_sims = 0, n_ev = 0;
    int err = 0, step = 0, done = 0;
    for (int i = 0; i < E; i++) {
        init_root(&trees[i].nodes[0], cfg->init_bb0, cfg->init_bb1, cfg->init_player);
        trees[i].used = 1;
    }
    while (!done && !err) {
        if (step >= cfg->max_steps) break;
        err = run_sims_noise(trees, E, S, cfg->c_puct, cfg->eval_kind, cb, user, &n_ev, eps, eta ? &eta[(size_t)step * E * 7] : NULL);
        if (err) break;
        n_sims += (int64_t)E * S;
        for (int i = 0; i < E; i++) {
            tree_t *t = &trees[i];
            node_t *r = &t->nodes[0];
            int l = h_len[i];
            if (l >= 42) { err = 6; break; }
            size_t o = (size_t)i * 42 + l;
            bb_from_cells(r->cell, &h_bb0[o], &h_bb1[o]);
            h_pl[o] = r->player;
            for (int c = 0; c < 7; c++) h_cnt[o * 7 + c] = 0;
            for (int j = 0; j < r->nchild; j++) {
                node_t *ch = &t->nodes[r->first_child + j];
                h_cnt[o * 7 + ch->col] = ch->N;
            }
            h_len[i] = l + 1;
            const double u = uniforms[(size_t)step * E + i];
            int j = (greedy_from >= 0 && l >= greedy_from) ? greedy_child(t) : sample_child(t, u);
            n_u++;
            node_t next = t->nodes[r->first_child + j];
            if (!next.ended) {
                next.parent = -1; next.first_child = -1; next.nchild = 0; next.N = 0; next.W = 0.0; next.P = 0.0;
                t->nodes[0] = next; t->used = 1;
                continue;
            }
            if (n_s + h_len[i] > max_samples) { err = 7; break; }
            ep_slot[n_ep] = i; ep_len[n_ep] = h_len[i]; ep_step[n_ep] = step;
            ep_outcome[2 * n_ep] = next.reward0; ep_outcome[2 * n_ep + 1] = (int8_t)-next.reward0;
            for (int k = 0; k < h_len[i]; k++) {
                size_t q = (size_t)i * 42 + k;
                s_bb0[n_s] = h_bb0[q]; s_bb1[n_s] = h_bb1[q]; s_player[n_s] = h_pl[q];
                memcpy(&s_counts[n_s * 7], &h_cnt[q * 7], sizeof(int32_t) * 7);
                n_s++;
            }
            n_ep++;
            h_len[i] = 0;
            init_root(&t->nodes[0], cfg->init_bb0, cfg->init_bb1, cfg->init_player);
            t->used = 1;
            if (n_ep >= cfg->quota) { done = 1; break; }
        }
        step++;
    }
    *n_episodes_out = n_ep; *n_samples_out = n_s; *n_steps_out = step; *n_uniforms_used = n_u;
    *n_sims_out = n_sims; *n_evals_out = n_ev;
    free(h_bb0); free(h_bb1); free(h_pl); free(h_cnt); free(h_len);
    free_trees(trees, E);
    return err;
}
