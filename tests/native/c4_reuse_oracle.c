/*
 * TEST INFRASTRUCTURE — the library's opt-in subtree reuse (az_set_subtree_reuse, AlphaGo Zero's "the child node corresponding
 * to the played action becomes the new root node; the subtree below this child is retained along with all its statistics")
 * restated on top of the noise oracle (tests/native/c4_noise_oracle.c, which includes oracle/c4_oracle.c; both included
 * unchanged).  The reference discards its tree after every move (node.py:37-41), so there are no goldens:
 * tests/test_oracle_subtree_reuse.py pins this file to c4o_selfplay_noise (V = S never retains anything) and to a walk of the
 * trees by column paths.
 *
 * Only what reuse adds is written here:
 *   - the retention rule: after the move to child c, if c is expanded and N(c) + S <= V the subtree of c becomes the tree;
 *     if c was never expanded ("fresh") or N(c) + S > V ("dropped") the tree is a fresh root; a finished game is recycled;
 *   - reroot(): the subtree of c compacted in place by one ascending sweep - the retained nodes keep their relative order
 *     (so c becomes node 0 and every children block stays contiguous), parent / first_child are remapped, and the new root's
 *     prior is 0 (N(c) and W(c) are kept);
 *   - trees are allocated for 1 + 7 V nodes: expand() fails (error 4) if a search ever needs more.
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (tests/reuse_oracle.py, into a temporary directory).
 */
#include "c4_noise_oracle.c"

enum { RO_RETAINED, RO_FRESH, RO_DROPPED, RO_NODES, RO_VISITS, RO_MAX_USED, RO_N };

/* the subtree of node c (c >= 1) becomes the tree, in place */
static int reroot(tree_t *t, int c) {
    int32_t *map = malloc(sizeof(int32_t) * (size_t)t->used);
    if (!map) return -1;
    for (int i = 0; i < t->used; i++) map[i] = -1;
    map[c] = 0;
    int n = 1;
    for (int i = c + 1; i < t->used; i++) {
        const int p = t->nodes[i].parent;
        if (p >= 0 && map[p] >= 0) map[i] = n++;
    }
    for (int i = c; i < t->used; i++) {
        if (map[i] < 0) continue;
        node_t nd = t->nodes[i];
        nd.parent = i == c ? -1 : map[nd.parent];
        nd.first_child = nd.nchild ? map[nd.first_child] : -1;
        if (i == c) nd.P = 0.0;
        t->nodes[map[i]] = nd; /* map[i] <= i: the source is read before anything overwrites it */
    }
    t->used = n;
    free(map);
    return 0;
}

static void fresh_root(tree_t *t, const node_t *c) {
    node_t r = *c;
    r.parent = -1; r.first_child = -1; r.nchild = 0; r.N = 0; r.W = 0.0; r.P = 0.0;
    t->nodes[0] = r;
    t->used = 1;
}

/* the move to node c of a game that goes on */
static int keep_subtree(tree_t *t, int c, int S, int V, int64_t *st) {
    const node_t *ch = &t->nodes[c];
    if (ch->nchild == 0) { st[RO_FRESH]++; fresh_root(t, ch); return 0; }
    if (ch->N + S > V) { st[RO_DROPPED]++; fresh_root(t, ch); return 0; }
    const int32_t visits = ch->N;
    if (reroot(t, c)) return 1;
    st[RO_RETAINED]++; st[RO_NODES] += t->used; st[RO_VISITS] += visits;
    return 0;
}

static void note_used(const tree_t *trees, int E, int64_t *st) {
    for (int i = 0; i < E; i++)
        if (trees[i].used > st[RO_MAX_USED]) st[RO_MAX_USED] = trees[i].used;
}

/* the tree of slot i in the engine's export format (az_export_tree): node 0 = root, first child 0 = none */
static void export_tree(const tree_t *t, int cap, double *W, uint32_t *N, float *P, uint32_t *CB) {
    for (int i = 0; i < cap; i++) { W[i] = 0.0; N[i] = 0; P[i] = 0.0f; CB[i] = 0; }
    for (int i = 0; i < t->used; i++) {
        const node_t *nd = &t->nodes[i];
        W[i] = nd->W; N[i] = (uint32_t)nd->N; P[i] = (float)nd->P; CB[i] = nd->nchild ? (uint32_t)nd->first_child : 0u;
    }
}

/* S1 simulations on E roots, the move cols[i] on every root (status[i] = 1 and the tree untouched for an illegal column; a move
 * that ends the game leaves a fresh root there, as the engine does), S2 more simulations, then the trees of the slots
 * export_slots[0 .. n_export) in the export format ([n_export][cap] arrays, cap >= 1 + 7 V) and their node counts.  st[RO_N]. */
int c4o_advance_reuse(int E, const uint64_t *bb0, const uint64_t *bb1, const uint8_t *player, int S1, int S2, int S, int V,
                      double c_puct, int eval_kind, c4o_eval_cb cb, void *user, const uint8_t *cols, uint8_t *status, int n_export,
                      const int32_t *export_slots, int cap, double *W, uint32_t *N, float *P, uint32_t *CB, int32_t *used,
                      int64_t *st) {
    tree_t *trees = alloc_trees(E, V);
    if (!trees || cap < trees[0].cap) return 1;
    for (int i = 0; i < E; i++) { init_root(&trees[i].nodes[0], bb0[i], bb1[i], player[i]); trees[i].used = 1; }
    for (int k = 0; k < RO_N; k++) st[k] = 0;
    int64_t ev = 0;
    int err = run_sims(trees, E, S1, c_puct, eval_kind, cb, user, &ev);
    note_used(trees, E, st);
    for (int i = 0; i < E && !err; i++) {
        tree_t *t = &trees[i];
        node_t *r = &t->nodes[0];
        const uint8_t lg = legal_mask_of(r);
        status[i] = 1;
        if (cols[i] >= Wd || !(lg >> cols[i] & 1)) continue;
        status[i] = 0;
        if (r->nchild == 0) { /* never searched: the root just moves on */
            node_t next;
            memset(&next, 0, sizeof next);
            play_into(r, cols[i], &next);
            fresh_root(t, &next);
            continue;
        }
        const int c = r->first_child + __builtin_popcount(lg & ((1u << cols[i]) - 1u));
        if (t->nodes[c].ended) { fresh_root(t, &t->nodes[c]); continue; }
        err = keep_subtree(t, c, S, V, st);
    }
    /* roots that ended cannot be searched (error 3 in the oracle, AZ_TREE_ROOT_ENDED in the engine): search the others */
    if (!err && S2 > 0) {
        int n_live = 0;
        tree_t *live = calloc(E > 0 ? (size_t)E : 1, sizeof *live);
        for (int i = 0; i < E; i++) if (!trees[i].nodes[0].ended) live[n_live++] = trees[i];
        err = run_sims(live, n_live, S2, c_puct, eval_kind, cb, user, &ev);
        for (int i = 0, j = 0; i < E; i++) if (!trees[i].nodes[0].ended) trees[i] = live[j++];
        free(live);
        note_used(trees, E, st);
    }
    for (int k = 0; k < n_export && !err; k++) {
        const int s = export_slots[k];
        export_tree(&trees[s], cap, &W[(size_t)k * cap], &N[(size_t)k * cap], &P[(size_t)k * cap], &CB[(size_t)k * cap]);
        used[k] = trees[s].used;
    }
    free_trees(trees, E);
    return err;
}

/* c4o_selfplay_noise (same loop, same outputs) with subtree reuse under max_root_visits V (>= S); st[RO_N] */
int c4o_selfplay_reuse(const c4o_selfplay_cfg *cfg, int V, const double *uniforms, c4o_eval_cb cb, void *user, float eps,
                       const float *eta, int greedy_from, int32_t *ep_slot, int32_t *ep_len, int32_t *ep_step,
                       int8_t *ep_outcome, uint64_t *s_bb0, uint64_t *s_bb1, uint8_t *s_player, int32_t *s_counts,
                       int64_t max_samples, int64_t *n_episodes_out, int64_t *n_samples_out, int64_t *n_steps_out,
                       int64_t *n_uniforms_used, int64_t *n_sims_out, int64_t *n_evals_out, int64_t *st) {
    int E = cfg->E, S = cfg->S;
    if (V < S) return 1;
    tree_t *trees = alloc_trees(E, V);
    if (!trees) return 1;
    uint64_t *h_bb0 = malloc(8 * (size_t)E * 42), *h_bb1 = malloc(8 * (size_t)E * 42);
    uint8_t *h_pl = malloc((size_t)E * 42);
    int32_t *h_cnt = malloc(sizeof(int32_t) * (size_t)E * 42 * 7);
    int *h_len = calloc((size_t)E, sizeof(int));
    int64_t n_ep = 0, n_s = 0, n_u = 0, n_sims = 0, n_ev = 0;
    int err = 0, step = 0, done = 0;
    for (int k = 0; k < RO_N; k++) st[k] = 0;
    for (int i = 0; i < E; i++) {
        init_root(&trees[i].nodes[0], cfg->init_bb0, cfg->init_bb1, cfg->init_player);
        trees[i].used = 1;
    }
    while (!done && !err) {
        if (step >= cfg->max_steps) break;
        err = run_sims_noise(trees, E, S, cfg->c_puct, cfg->eval_kind, cb, user, &n_ev, eps, eta ? &eta[(size_t)step * E * 7] : NULL);
        if (err) break;
        note_used(trees, E, st);
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
                err = keep_subtree(t, r->first_child + j, S, V, st);
                if (err) break;
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
