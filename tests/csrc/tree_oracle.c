/*
 * tests/csrc/tree_oracle.c -- TEST INFRASTRUCTURE: the CPU oracle's search, with its whole tree kept.
 *
 * Includes oracle/gmz_oracle.c unchanged and reuses every piece of it (Tree, select_leaf, backpropagate, the halving
 * schedule, sequential_halving, the decision); only the driver loop of orc_search is restated here, so that the tree
 * can be written out before it is freed.  tests/test_tree_export_cpu.py pins this loop to orc_search (visits, value,
 * action, policy, MinMax and leaf traces, bit for bit) and so to the reference goldens; tests/test_tree_export_gpu.py
 * compares the engine's gmz_tree_export against it node for node.  Built on demand by tests/_tree_oracle.py with the
 * oracle's own flags (-ffp-contract=off).
 */
#include "../../oracle/gmz_oracle.c"

/* Every pointer may be NULL.  Per node k < n_nodes (node 0 the root, node k the k-th created): arrays of num_simulations
 * entries, -1 / 0 past n_nodes.  Top-k arrays of num_top_actions entries in halving order (survivors first, each
 * halving's losers behind them), -1 / 0 past the initial top-k. */
typedef struct {
    int32_t *parent, *action, *depth, *visits;   /* -1 parent / action for the root */
    double *value_sum, *reward;
    float *prior_logit;                           /* the parent's logit at `action`, NaN for the root */
    int32_t *counts;                              /* [5] n_nodes, sim_count, current_phase, len(selected), n_init */
    double *minmax;                               /* [2] minimum, maximum */
    int32_t *topk_action, *topk_round;            /* round = the halving that eliminated the entry, current_phase if selected */
    double *topk_gumbel;
    float *topk_logit;
} tro_tree;

/* The initial top-k in halving order and the round each entry was eliminated in (-1 = still selected). */
typedef struct { int *act, *round; int n_init; } TopK;

/* _sequential_halving (mcts.py:183-185) through the oracle's own sequential_halving, keeping the eliminated entries:
 * with current_num_top_actions raised to len(selected) it keeps every entry, so `sel` holds the whole stable descending
 * order; the first `keep` of it are what the oracle keeps. */
static void halving_recorded(Tree *t, TopK *k, double *tq)
{
    const int n = t->n_sel, m = t->current_num_top_actions, keep = m < n ? m : n;
    t->current_num_top_actions = n;
    sequential_halving(t, tq);
    t->current_num_top_actions = m;
    for (int i = 0; i < n; ++i) k->act[i] = t->sel[i];
    for (int i = keep; i < n; ++i) k->round[i] = t->current_phase;
    t->n_sel = keep;
}

static void tree_write(const Tree *t, const TopK *k, const orc_config *cfg, int sim_count, const tro_tree *o)
{
    const int S = cfg->num_simulations, K = cfg->num_top_actions, n = t->n_nodes;
    int *dep = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
    for (int i = 0; i < S; ++i) {
        const Node *nd = i < n ? &t->nodes[i] : NULL;
        if (nd) dep[i] = nd->parent < 0 ? 0 : dep[nd->parent] + 1;     /* parents are created before their children */
        if (o->parent) o->parent[i] = nd ? nd->parent : -1;
        if (o->action) o->action[i] = nd ? nd->action : -1;
        if (o->depth) o->depth[i] = nd ? dep[i] : -1;
        if (o->visits) o->visits[i] = nd ? nd->visit_count : -1;
        if (o->value_sum) o->value_sum[i] = nd ? nd->value_sum : 0.0;
        if (o->reward) o->reward[i] = nd ? nd->reward : 0.0;
        if (o->prior_logit) o->prior_logit[i] = !nd ? 0.0f : nd->parent < 0 ? NAN : t->nodes[nd->parent].logits[nd->action];
    }
    free(dep);
    if (o->counts) { o->counts[0] = n; o->counts[1] = sim_count; o->counts[2] = t->current_phase; o->counts[3] = t->n_sel; o->counts[4] = k->n_init; }
    if (o->minmax) { o->minmax[0] = t->mm.minimum; o->minmax[1] = t->mm.maximum; }
    for (int i = 0; i < K; ++i) {
        const int in = i < k->n_init, a = in ? k->act[i] : -1;
        if (o->topk_action) o->topk_action[i] = a;
        if (o->topk_round) o->topk_round[i] = !in ? -1 : k->round[i] < 0 ? t->current_phase : k->round[i];
        if (o->topk_gumbel) o->topk_gumbel[i] = in ? t->gumbel[a] : 0.0;
        if (o->topk_logit) o->topk_logit[i] = in ? t->nodes[0].logits[a] : 0.0f;
    }
}

/* orc_search (gmz_oracle.c) with the tree written to `o` before it is freed; same arguments and outputs, the leaf
 * traces included.  The loop below is orc_search's, line for line, with sequential_halving -> halving_recorded. */
int tro_search_tree(const orc_config *cfg, const int8_t *board, int player, int last_move, int move_count,
                    const double *gumbel, double *out_policy, double *out_value, int32_t *out_action,
                    int32_t *out_visits, int32_t *out_leaf_actions, int32_t *out_leaf_depths, const tro_tree *o)
{
    const int A = cfg->board_size * cfg->board_size, S = cfg->num_simulations;
    uint8_t *valid = (uint8_t *)malloc((size_t)A);
    int n_valid = 0;
    for (int a = 0; a < A; ++a) { valid[a] = board[a] == 0; n_valid += valid[a]; }
    for (int a = 0; a < A; ++a) out_policy[a] = 0.0;
    *out_value = 0.0; *out_action = -1;
    if (out_visits) memset(out_visits, 0, sizeof(int32_t) * (size_t)A);
    Tree t; memset(&t, 0, sizeof(t));
    TopK k; memset(&k, 0, sizeof(k));
    if (n_valid == 0) {      /* the sentinel: no tree */
        mm_init(&t.mm, cfg->minmax_delta, 0);
        tree_write(&t, &k, cfg, 0, o);
        free(valid);
        return 1;
    }

    t.cfg = cfg; t.A = A; t.cap = S + 4; t.nodes = (Node *)malloc(sizeof(Node) * (size_t)t.cap);
    t.valid = valid; t.gumbel = gumbel; t.f32 = cfg->accum_dtype == 1; mm_init(&t.mm, cfg->minmax_delta, t.f32);
    float *logits = (float *)malloc(sizeof(float) * (size_t)A);
    double *tq = (double *)malloc(sizeof(double) * (size_t)A), *pol = (double *)malloc(sizeof(double) * (size_t)A);
    int8_t *tmp = (int8_t *)malloc((size_t)A);
    int *hist = (int *)malloc(sizeof(int) * (size_t)(S + 4));
    double value; uint64_t hidden;

    const int root = node_new(&t, -1, -1);
    orc_e0_initial(cfg, board, player, last_move, logits, &value, &hidden);
    node_expand(&t, root, logits, hidden, 0.0);
    backpropagate(&t, root, value);

    halving_init(&t);
    {
        double *sc = (double *)malloc(sizeof(double) * (size_t)n_valid); int *ac = (int *)malloc(sizeof(int) * (size_t)n_valid);
        int n = 0;
        for (int a = 0; a < A; ++a) if (valid[a]) { sc[n] = gumbel[a] + (double)t.nodes[root].logits[a]; ac[n] = a; ++n; }
        for (int i = 1; i < n; ++i) {
            double s = sc[i]; int a = ac[i]; int j = i - 1;
            while (j >= 0 && (sc[j] < s || (sc[j] == s && ac[j] < a))) { sc[j + 1] = sc[j]; ac[j + 1] = ac[j]; --j; }
            sc[j + 1] = s; ac[j + 1] = a;
        }
        t.n_sel = n < t.current_num_top_actions ? n : t.current_num_top_actions;
        t.sel = (int *)malloc(sizeof(int) * (size_t)(t.n_sel > 0 ? t.n_sel : 1));
        for (int i = 0; i < t.n_sel; ++i) t.sel[i] = ac[i];
        k.n_init = t.n_sel;
        k.act = (int *)malloc(sizeof(int) * (size_t)(t.n_sel > 0 ? t.n_sel : 1));
        k.round = (int *)malloc(sizeof(int) * (size_t)(t.n_sel > 0 ? t.n_sel : 1));
        for (int i = 0; i < t.n_sel; ++i) { k.act[i] = ac[i]; k.round[i] = -1; }
        free(sc); free(ac);
    }

    int sim_count = 1, n_evals = 0;
    while (sim_count < S) {
        int depth = 0;
        if (cfg->mode == 0) {
            int leaf = select_leaf(&t, tq, pol, &depth);
            int n_hist = 0;
            for (int nd = leaf; t.nodes[nd].parent >= 0; nd = t.nodes[nd].parent) hist[n_hist++] = t.nodes[nd].action;
            memcpy(tmp, board, (size_t)A);
            int p = player, lm = -1, mc = move_count;
            for (int i = n_hist - 1; i >= 0; --i) do_move(tmp, &p, &lm, &mc, hist[i]);
            orc_e0_initial(cfg, tmp, p, lm, logits, &value, &hidden);
            node_expand(&t, leaf, logits, hidden, 0.0);
            backpropagate(&t, leaf, value);
            if (out_leaf_actions) out_leaf_actions[n_evals] = t.nodes[leaf].action;
            if (out_leaf_depths) out_leaf_depths[n_evals] = depth;
            ++n_evals; sim_count += 1;
        } else {
            const int n = t.n_sel;
            if (n == 0) break;
            int leaf = -1;
            for (int i = 0; i < n; ++i) leaf = select_leaf(&t, tq, pol, &depth);
            double reward;
            const int parent = t.nodes[leaf].parent;
            orc_e0_recurrent(cfg, t.nodes[parent].hidden, t.nodes[leaf].action, logits, &value, &reward, &hidden);
            for (int i = 0; i < n; ++i) node_expand(&t, leaf, logits, hidden, reward);
            for (int i = 0; i < n; ++i) backpropagate(&t, leaf, value);
            if (out_leaf_actions) out_leaf_actions[n_evals] = t.nodes[leaf].action;
            if (out_leaf_depths) out_leaf_depths[n_evals] = depth;
            ++n_evals; sim_count += n;
        }
        if (halving_ready(&t, sim_count)) halving_recorded(&t, &k, tq);
    }

    transformed_qs(&t, root, tq);
    improved_policy(&t, root, tq, out_policy);
    *out_value = node_get_value(&t, &t.nodes[root]);
    {
        int32_t *keys = (int32_t *)malloc(sizeof(int32_t) * (size_t)n_valid), *order = (int32_t *)malloc(sizeof(int32_t) * (size_t)n_valid);
        int n = 0;
        for (int a = 0; a < A; ++a) if (valid[a]) keys[n++] = a;
        orc_pyset_order(keys, n_valid, order);
        int best = -1, best_n = -1;
        for (int i = 0; i < n_valid; ++i) {
            int ch = node_child_or_neg(&t, root, order[i]);
            int v = ch >= 0 ? t.nodes[ch].visit_count : 0;
            if (v > best_n) { best_n = v; best = order[i]; }
        }
        *out_action = best;
        free(keys); free(order);
    }
    if (out_visits)
        for (int a = 0; a < A; ++a) { int ch = node_child_or_neg(&t, root, a); out_visits[a] = ch >= 0 ? t.nodes[ch].visit_count : 0; }
    tree_write(&t, &k, cfg, sim_count, o);

    tree_free(&t); free(k.act); free(k.round); free(valid); free(logits); free(tq); free(pol); free(tmp); free(hist);
    return 0;
}
