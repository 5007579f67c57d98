/*
 * oracle_search.c -- TEST INFRASTRUCTURE (CPU oracle); see oracle.h.
 *
 * Symmetrizers, evaluators, the UCT tree and the self-play loop, restated from
 * symmetry/D4GridSymmetrizer.hpp, symmetry/ConnectFourSymmetrizer.cpp,
 * networks/{RandomNetwork,GridNetwork}.hpp, uct/UCTNode.hpp, uct/UCTTree.hpp
 * and selfplay/SelfPlay.hpp.  fp32 expressions keep the reference's operand
 * order; compile with -ffp-contract=off.
 */
#include "oracle_internal.h"

#include <stdio.h>

/* ------------------------------------------------------------ symmetrizers */
/* symmetry/D4GridSymmetrizer.hpp:106-117: new[f_s(r,c)] = old[r,c] */
static void d4_map(int w, int sym, int r, int c, int* tr, int* tc) {
    switch (sym) {
    case 0: *tr = r; *tc = c; break;
    case 1: *tr = c; *tc = w - 1 - r; break;
    case 2: *tr = w - 1 - r; *tc = w - 1 - c; break;
    case 3: *tr = w - 1 - c; *tc = r; break;
    case 4: *tr = r; *tc = w - 1 - c; break;
    case 5: *tr = w - 1 - c; *tc = w - 1 - r; break;
    case 6: *tr = w - 1 - r; *tc = c; break;
    default: *tr = c; *tc = r; break;
    }
}

static int sym_cell(int game, int sym, int from) {
    const ogame_info* gi = og_info(game);
    int r = from / gi->cols, c = from % gi->cols, tr, tc;
    if (game == OG_C4) {    /* symmetry/ConnectFourSymmetrizer.cpp:17-56: 1 = column flip */
        return sym == 1 ? r * 7 + (6 - c) : from;
    }
    d4_map(gi->cols, sym, r, c, &tr, &tc);
    return tr * gi->cols + tc;
}

void osym_cells(int game, int sym, const int8_t* in, int8_t* out) {
    const ogame_info* gi = og_info(game);
    for (int i = 0; i < gi->cells; ++i) out[sym_cell(game, sym, i)] = in[i];
}

void osym_dist(int game, int sym, const float* in, float* out) {
    const ogame_info* gi = og_info(game);
    if (game == OG_C4) {    /* symmetry/ConnectFourSymmetrizer.cpp:60-99: actions are columns */
        for (int c = 0; c < 7; ++c) out[sym == 1 ? 6 - c : c] = in[c];
        return;
    }
    for (int i = 0; i < gi->cells; ++i) out[sym_cell(game, sym, i)] = in[i];
    out[gi->cells] = in[gi->cells];     /* pass stays put, symmetry/D4GridSymmetrizer.hpp:94-95 */
}

int osym_inverse(int game, int sym) {
    static const int inv[8] = { 0, 3, 2, 1, 4, 5, 6, 7 };   /* symmetry/D4GridSymmetrizer.hpp:47-50 */
    return game == OG_C4 ? sym : inv[sym];
}

void oracle_symmetrize_cells(int game, int sym, const int8_t* in, int8_t* out) { osym_cells(game, sym, in, out); }
void oracle_symmetrize_dist(int game, int sym, const float* in, float* out) { osym_dist(game, sym, in, out); }
int oracle_inverse_symmetry(int game, int sym) { return osym_inverse(game, sym); }

/* -------------------------------------------------------------- evaluators */
typedef struct {
    int8_t hist[OG_MAXH][OG_MAXB];
    int size;
    int player;
} ostate;

/* Network input planes, networks/GridNetwork.hpp:72-97 (same as the sample
 * embedding of selfplay/GridWorker.hpp:146-171). */
static void embed_state(const ogame_info* gi, const ostate* s, float* planes) {
    int B = gi->cells, own = s->player, opp = 1 - own;
    for (int t = 0; t < gi->history; ++t) {
        for (int i = 0; i < B; ++i) {
            planes[(2 * t) * B + i] = (t < s->size && s->hist[t][i] == own) ? 1.0f : 0.0f;
            planes[(2 * t + 1) * B + i] = (t < s->size && s->hist[t][i] == opp) ? 1.0f : 0.0f;
        }
    }
    for (int i = 0; i < B; ++i) planes[2 * gi->history * B + i] = (s->player == O_ZERO) ? 1.0f : 0.0f;
}

static float dist_sum(const float* d, int n) {      /* games/GameActionDist.hpp:87-95 */
    float r = 0.0f;
    for (int i = 0; i < n; ++i) r += d[i];
    return r;
}
static void dist_div(float* d, int n, float rhs) {  /* games/GameActionDist.hpp:283-293 */
    float inv = 1.0f / rhs;
    for (int i = 0; i < n; ++i) d[i] = d[i] * inv;
}

/* mask -> sum -> normalise tail of networks/GridNetwork.hpp:117-139 */
static void mask_normalise(float* policy, const float* mask, int A) {
    int numLegal = 0;
    for (int i = 0; i < A; ++i) {
        if (mask[i] == 0.0f) policy[i] = 0.0f; else ++numLegal;
    }
    float sum = dist_sum(policy, A);
    if (sum == 0.0f) {
        float uniform = 1.0f / numLegal;
        for (int i = 0; i < A; ++i) policy[i] = (mask[i] == 0.0f) ? 0.0f : uniform;
    } else {
        dist_div(policy, A, sum);
    }
}

static void hashnet_eval(const ogame_info* gi, const ostate* s, const float* mask, uint64_t salt, float* policy, float* value) {
    uint64_t words[4 * OG_MAXH];
    memset(words, 0, sizeof(words));
    int own = s->player, opp = 1 - own;
    for (int t = 0; t < s->size; ++t)
        for (int i = 0; i < gi->cells; ++i) {
            if (s->hist[t][i] == own) words[4 * t + (i >> 6)] |= 1ULL << (i & 63);
            if (s->hist[t][i] == opp) words[4 * t + 2 + (i >> 6)] |= 1ULL << (i & 63);
        }
    uint64_t h = ohashnet_salt(ohashnet_state_hash(words, s->size, s->player), salt);
    for (int i = 0; i < gi->actions; ++i) policy[i] = ohashnet_prior_raw(h, i);
    mask_normalise(policy, mask, gi->actions);
    *value = ohashnet_value(h);
}

void oracle_hashnet(int game, const int8_t* hist_cells, int hist_size, int player, const float* mask,
                    float* policy, float* value) {
    const ogame_info* gi = og_info(game);
    ostate s;
    memset(&s, 0, sizeof(s));
    for (int t = 0; t < hist_size; ++t) memcpy(s.hist[t], hist_cells + t * gi->cells, (size_t)gi->cells);
    s.size = hist_size;
    s.player = player;
    hashnet_eval(gi, &s, mask, 0, policy, value);
}

/* INetwork::evaluate for a batch (networks/INetwork.hpp:25-27) */
static void evaluate_batch(const oracle_selfplay_cfg* cfg, const ogame_info* gi, const ostate* states,
                           const float (*masks)[OG_MAXA], int n, float (*policy)[OG_MAXA], float* value) {
    int A = gi->actions;
    if (cfg->evaluator == OE_UNIFORM) {          /* networks/RandomNetwork.hpp:21-49 */
        for (int b = 0; b < n; ++b) {
            int numLegal = 0;
            for (int i = 0; i < A; ++i) if (masks[b][i] > 0.0f) ++numLegal;
            float uniform = 1.0f / numLegal;
            for (int i = 0; i < A; ++i) policy[b][i] = (masks[b][i] > 0.0f) ? uniform : 0.0f;
            value[b] = 0.0f;
        }
    } else if (cfg->evaluator == OE_HASHNET) {
        for (int b = 0; b < n; ++b) hashnet_eval(gi, &states[b], masks[b], cfg->hash_salt, policy[b], &value[b]);
    } else if (cfg->evaluator == OE_HEURISTIC) { /* networks/OthelloHeuristic.cpp:5-53 */
        for (int b = 0; b < n; ++b) {
            int numLegal = 0, numEmpty = 0, numOppLegal = 0;
            for (int i = 0; i < A; ++i) if (masks[b][i] > 0.0f) ++numLegal;      /* counts the pass slot too */
            float uniform = 1.0f / numLegal;
            for (int i = 0; i < A; ++i) policy[b][i] = (masks[b][i] > 0.0f) ? uniform : 0.0f;
            for (int i = 0; i < gi->cells; ++i) if (states[b].hist[0][i] == O_NONE) ++numEmpty;
            float oppMask[OG_MAXA];
            og_othello_mask(states[b].hist[0], 1 - states[b].player, oppMask);
            for (int i = 0; i < gi->cells; ++i) if (oppMask[i] > 0.0f) ++numOppLegal;   /* placements only */
            value[b] = (float)(numLegal - numOppLegal) / numEmpty;
        }
    } else {                                     /* networks/GridNetwork.hpp:62-145 */
        int plane = (2 * gi->history + 1) * gi->cells;
        float* planes = (float*)malloc(sizeof(float) * (size_t)plane * (size_t)n);
        float* logits = (float*)malloc(sizeof(float) * (size_t)A * (size_t)n);
        for (int b = 0; b < n; ++b) embed_state(gi, &states[b], planes + (size_t)b * plane);
        cfg->eval_cb(cfg->eval_user, planes, n, logits, value);
        for (int b = 0; b < n; ++b) {
            for (int i = 0; i < A; ++i) policy[b][i] = odet_expf(logits[(size_t)b * A + i]);
            mask_normalise(policy[b], masks[b], A);
        }
        free(planes);
        free(logits);
    }
}

/* --------------------------------------------------------------- UCT tree */
typedef struct {
    const oracle_selfplay_cfg* cfg;
    const ogame_info* gi;
    int game;
    orng_t* rng;
    onode* game_root;       /* m_gameRoot / m_uctRoot */
    onode* decision;        /* m_decisionNode */
    float root_P[1], root_W[1], root_N[1];   /* tree-level dummy edge, uct/UCTTree.hpp:301 (action 0) */
    oracle_selfplay_out* stats;
    oracle_search_stats* search;    /* may be NULL */
    int last_depth;         /* edges of the last descent (search stats only) */
} otree;

static void node_attach_stats(onode* n) {
    /* child ctor: m_parentEdgeStatistics = &parent->m_edgeStatistics (uct/UCTNode.hpp:90-97) */
    n->own_N = &n->parent->N[n->action];
    n->own_W = &n->parent->W[n->action];
}

/* uct/UCTNode.hpp:258-284 */
static onode* uct_get_add_child(otree* t, onode* n, int action) {
    if (!n->child[action]) {
        onode* c = og_get_add_child(t->game, n, action);
        node_attach_stats(c);
        if (t->cfg->init_q == OQ_PARENT) n->W[action] = n->evaluated ? n->net_value : 0.0f;
        else n->W[action] = 0.0f;           /* ZERO, and DROP_PARENT ("never used", :273-278) */
    }
    return n->child[action];
}

/* UCTNode::Q, uct/UCTNode.hpp:152-163.  With DROP_PARENT an unvisited node answers with its parent's Q; the
 * decision node keeps its predecessor as m_parent, so the walk never leaves the tree. */
static float uct_node_q(otree* t, onode* n) {
    if (t->cfg->init_q == OQ_DROP_PARENT) {
        if (*n->own_N == 0) return n->parent ? uct_node_q(t, n->parent) : 0.0f;   /* root of a fresh tree: null deref in the reference */
        return *n->own_W / *n->own_N;
    }
    return *n->own_W / (1 + *n->own_N);
}

/* uct/UCTNode.hpp:221-251 with child_Q / child_U of :191-211 */
static int uct_best_action(otree* t, onode* n) {
    int A = t->gi->actions, nbest = 0;
    int best[OG_MAXA];
    float bestValue = -__builtin_inff();
    float uWeight = t->cfg->u_weight;
    for (int a = 0; a < A; ++a) {
        if (n->mask[a] == 0.0f) continue;
        float q;
        if (t->cfg->init_q == OQ_DROP_PARENT) q = (n->N[a] == 0) ? uct_node_q(t, n) : n->W[a] / n->N[a];
        else q = n->W[a] / (1 + n->N[a]);
        float u = n->P[a] * __builtin_sqrtf(*n->own_N) / (1 + n->N[a]);
        float value = q + uWeight * u;
        if (value > bestValue) { bestValue = value; nbest = 0; best[nbest++] = a; }
        else if (value == bestValue) best[nbest++] = a;
    }
    return best[orng_uniform_int(t->rng, 0, nbest - 1)];
}

/* uct/UCTNode.hpp:314-348 */
static void uct_expand(otree* t, onode* n, int addNoise) {
    int A = t->gi->actions, numLegal = 0;
    n->expanded = 1;
    for (int a = 0; a < A; ++a) {
        if (n->mask[a] == 0.0f) continue;
        n->P[a] = n->net_policy[a];
        ++numLegal;
    }
    if (addNoise) {
        float noise[OG_MAXA];
        float eps = t->cfg->dir_eps;
        orng_dirichlet(t->rng, t->cfg->dir_alpha, noise, numLegal);
        int k = 0;
        for (int a = 0; a < A; ++a) {
            if (n->mask[a] == 0.0f) continue;
            /* (1.0 - m_dirEps) * P + m_dirEps * noise: double * float + (float * float) */
            n->P[a] = (float)((1.0 - (double)eps) * (double)n->P[a] + (double)(eps * noise[k]));
            ++k;
        }
    }
}

/* uct/UCTTree.hpp:225-249 */
static onode* tree_select_leaf(otree* t) {
    onode* cur = t->decision;
    int depth = 0;
    while (cur->expanded && !cur->terminal) {
        int a = uct_best_action(t, cur);
        if (t->stats || t->search) {
            int nl = 0;
            for (int i = 0; i < t->gi->actions; ++i) nl += cur->mask[i] != 0.0f;
            if (t->stats) {
                t->stats->select_legal_sum += nl;
                t->stats->select_nodes += 1;
            }
            if (t->search) t->search->select_legal_sum += nl;
        }
        *cur->own_N += 1;
        *cur->own_W -= 1;
        cur = uct_get_add_child(t, cur, a);
        ++depth;
    }
    *cur->own_N += 1;
    *cur->own_W -= 1;
    if (t->stats) t->stats->select_depth_sum += depth;
    t->last_depth = depth;
    return cur;
}

/* uct/UCTTree.hpp:261-273 */
static void tree_backup(otree* t, onode* node, float valueEstimate) {
    float estimate = -valueEstimate * ((node->player == O_ZERO) ? 1 : -1);
    onode* cur = node;
    onode* stop = t->decision->parent;
    while (cur != stop) {
        *cur->own_W += 1 + estimate * ((cur->player == O_ZERO) ? 1 : -1);
        cur = cur->parent;
    }
}

/* search stats: the last descent ended at a leaf handled as `kind` (0 terminal, 1 gray, 2 queued as entry `k` of
 * `leaves`) */
static void note_descent(otree* t, int kind, onode** leaves, int k) {
    oracle_search_stats* s = t->search;
    if (!s) return;
    int d = t->last_depth;
    s->select_depth_sum += d;
    if (d > s->select_depth_max) s->select_depth_max = d;
    s->depth_hist[d < ODEPTH_BINS - 1 ? d : ODEPTH_BINS - 1] += 1;
    if (kind == 0) s->leaves_terminal += 1;
    else if (kind == 1) s->leaves_gray += 1;
    else s->leaves_empty += 1;
    if (d >= 32) {
        if (kind == 0) s->deep_terminal += 1;
        else if (kind == 1) s->deep_gray += 1;
        else s->deep_queued += 1;
    }
    if (kind == 2) {
        if (k + 1 > s->queue_max) s->queue_max = k + 1;
        for (int j = 0; j < k; ++j) {
            if (leaves[j] != leaves[k]) continue;
            s->dup_total += 1;
            if (k < 32) s->dup_first32 += 1;
            break;
        }
    }
}

/* uct/UCTTree.hpp:76-114 */
static int tree_search(otree* t, onode** leaves, int* nleaves) {
    int traversals = 0;
    *nleaves = 0;
    while (traversals < t->cfg->max_batch) {
        ++traversals;
        onode* leaf = tree_select_leaf(t);
        if (leaf->terminal) {
            float rewards[2];
            og_rewards(leaf, rewards);
            tree_backup(t, leaf, rewards[leaf->player]);
            if (t->stats) t->stats->leaves_terminal++;
            note_descent(t, 0, leaves, 0);
            continue;
        } else if (leaf->evaluated) {
            uct_expand(t, leaf, t->cfg->add_noise && leaf == t->decision);
            tree_backup(t, leaf, leaf->net_value);
            if (t->stats) t->stats->leaves_gray++;
            note_descent(t, 1, leaves, 0);
            continue;
        } else {
            leaves[(*nleaves)++] = leaf;
            if (t->stats) t->stats->leaves_empty++;
            note_descent(t, 2, leaves, *nleaves - 1);
        }
        if (*nleaves >= t->cfg->max_queue) break;
    }
    return traversals;
}

/* uct/UCTTree.hpp:124-184 */
static void tree_evaluate_and_backprop(otree* t, onode** leaves, int n) {
    const ogame_info* gi = t->gi;
    ostate* states = (ostate*)calloc((size_t)n, sizeof(ostate));
    float (*masks)[OG_MAXA] = calloc((size_t)n, sizeof(*masks));
    float (*policy)[OG_MAXA] = calloc((size_t)n, sizeof(*policy));
    float* value = (float*)calloc((size_t)n, sizeof(float));
    int* syms = (int*)calloc((size_t)n, sizeof(int));
    for (int i = 0; i < n; ++i) {
        states[i].size = og_game_state(t->game, leaves[i], states[i].hist);
        states[i].player = leaves[i]->player;
        memcpy(masks[i], leaves[i]->mask, sizeof(float) * OG_MAXA);    /* NOT symmetrised: quirk Q3 */
    }
    if (t->cfg->use_sym) {
        for (int i = 0; i < n; ++i) {
            syms[i] = orng_uniform_int(t->rng, 0, gi->nsym - 1);
            ostate s = states[i];
            for (int h = 0; h < s.size; ++h) osym_cells(t->game, syms[i], s.hist[h], states[i].hist[h]);
            if (t->cfg->fix_symmetry_mask) {        /* option, not the reference: the mask follows the state */
                float m[OG_MAXA];
                memcpy(m, masks[i], sizeof(m));
                osym_dist(t->game, syms[i], m, masks[i]);
            }
        }
    }
    evaluate_batch(t->cfg, gi, states, (const float (*)[OG_MAXA])masks, n, policy, value);
    if (t->stats) t->stats->total_evals += n;
    if (t->search) t->search->total_evals += n;
    for (int i = 0; i < n; ++i) {
        onode* leaf = leaves[i];
        float pol[OG_MAXA];
        memcpy(pol, policy[i], sizeof(pol));
        if (t->cfg->use_sym) osym_dist(t->game, osym_inverse(t->game, syms[i]), policy[i], pol);
        if (!leaf->evaluated) {         /* uct/UCTNode.hpp:292-301 */
            leaf->evaluated = 1;
            memcpy(leaf->net_policy, pol, sizeof(float) * (size_t)gi->actions);
            leaf->net_value = value[i];
        }
        if (!leaf->expanded) uct_expand(t, leaf, t->cfg->add_noise && leaf == t->decision);
        tree_backup(t, leaf, leaf->net_value);
    }
    free(states); free(masks); free(policy); free(value); free(syms);
}

/* uct/UCTTree.hpp:283-298 */
static void tree_clear_subtree(otree* t, onode* n) {
    if (!n->expanded) return;
    for (int a = 0; a < OG_MAXA; ++a) { n->P[a] = 0.0f; n->W[a] = 0.0f; n->N[a] = 0.0f; }
    n->expanded = 0;
    for (int a = 0; a < t->gi->actions; ++a)
        if (n->child[a]) tree_clear_subtree(t, n->child[a]);
}

/* uct/UCTTree.hpp:197-210 */
static void tree_advance(otree* t, int action) {
    og_prune_children_except(t->decision, action, t->gi->actions);
    onode* child = uct_get_add_child(t, t->decision, action);
    tree_clear_subtree(t, child);
    t->decision = child;
}

/* ------------------------------------------------------------------ selfPlay */
#define PUT(arr, idx, val) do { if (arr) (arr)[idx] = (val); } while (0)

/* selfplay/SelfPlay.hpp:50-192 for one game; appends to `out` */
static int self_play_game(const oracle_selfplay_cfg* cfg, uint64_t game_id, int gslot, oracle_selfplay_out* out,
                          oracle_search_stats* search) {
    const ogame_info* gi = og_info(cfg->game);
    int A = gi->actions, B = gi->cells, S = cfg->use_sym ? gi->nsym : 1;
    int plane = (2 * gi->history + 1) * B;
    orng_t rng = { cfg->seed, game_id, 0 };
    otree t;
    memset(&t, 0, sizeof(t));
    t.cfg = cfg; t.gi = gi; t.game = cfg->game; t.rng = &rng; t.stats = out; t.search = search;
    t.game_root = og_new_root(cfg->game);
    t.game_root->own_N = &t.root_N[0];
    t.game_root->own_W = &t.root_W[0];
    t.decision = t.game_root;

    int64_t sample0 = out->n_samples;
    int8_t* players = (int8_t*)malloc(4096);
    int moveCount = 0;
    onode** leaves = (onode**)malloc(sizeof(onode*) * (size_t)(cfg->max_batch > 0 ? cfg->max_batch : 1));
    int rc = 0;

    while (!t.decision->terminal) {
        if (out->n_moves >= out->cap_moves || out->n_samples + S > out->cap_samples || moveCount >= 4096) { rc = -1; break; }
        onode* root = t.decision;
        ostate st;
        memset(&st, 0, sizeof(st));
        st.size = og_game_state(cfg->game, root, st.hist);
        st.player = root->player;
        /* symmetrised sample states, order s = 0..S-1 (selfplay/SelfPlay.hpp:86-96) */
        for (int s = 0; s < S; ++s) {
            ostate ss = st;
            if (cfg->use_sym) for (int h = 0; h < st.size; ++h) osym_cells(cfg->game, s, st.hist[h], ss.hist[h]);
            if (out->states) embed_state(gi, &ss, out->states + (size_t)(out->n_samples + s) * plane);
        }
        int64_t evals0 = out->total_evals;
        int traversals = 0;
        while (traversals < cfg->sims) {            /* selfplay/SelfPlay.hpp:99-108 */
            int nleaves = 0;
            int trav = tree_search(&t, leaves, &nleaves);
            if (nleaves > 0) tree_evaluate_and_backprop(&t, leaves, nleaves);
            traversals += trav;
        }
        out->total_traversals += traversals;
        if (search) search->total_traversals += traversals;

        int64_t m = out->n_moves;
        for (int a = 0; a < A; ++a) {
            PUT(out->move_N, m * A + a, root->N[a]);
            PUT(out->move_W, m * A + a, root->W[a]);
            PUT(out->move_P, m * A + a, root->P[a]);
        }
        PUT(out->move_root_N, m, *root->own_N);
        PUT(out->move_root_W, m, *root->own_W);
        PUT(out->move_traversals, m, traversals);
        PUT(out->move_evals, m, (int32_t)(out->total_evals - evals0));
        PUT(out->move_player, m, root->player);
        if (out->move_board) memcpy(out->move_board + m * B, root->cells, (size_t)B);

        /* visits -> pdf -> pow -> pdf -> cdf (selfplay/SelfPlay.hpp:111-125) */
        float pdf[OG_MAXA], cdf[OG_MAXA];
        memcpy(pdf, root->N, sizeof(float) * (size_t)A);
        dist_div(pdf, A, dist_sum(pdf, A));
        float e = (moveCount < 15) ? 0.98f : 10.0f;     /* constants.hpp:8-10 */
        for (int a = 0; a < A; ++a) pdf[a] = odet_powf(pdf[a], e);
        dist_div(pdf, A, dist_sum(pdf, A));
        cdf[0] = pdf[0];
        for (int a = 1; a < A; ++a) cdf[a] = cdf[a - 1] + pdf[a];
        dist_div(cdf, A, cdf[A - 1]);
        for (int s = 0; s < S; ++s) {
            if (!out->distributions) break;
            float* dst = out->distributions + (size_t)(out->n_samples + s) * A;
            if (cfg->use_sym) osym_dist(cfg->game, s, pdf, dst); else memcpy(dst, pdf, sizeof(float) * (size_t)A);
        }
        int action;
        if (cfg->caller_moves) {                    /* std::max_element: the first action with the most visits */
            action = 0;
            for (int a = 1; a < A; ++a) if (root->N[a] > root->N[action]) action = a;
        } else {
            action = orng_sample_cdf(&rng, cdf, A);
        }
        PUT(out->move_action, m, action);
        players[moveCount] = root->player;
        tree_advance(&t, action);
        ++moveCount;
        out->n_moves += 1;
        out->n_samples += S;
    }

    if (rc == 0) {
        float rewards[2];
        og_rewards(t.decision, rewards);
        if (out->outcomes)
            for (int mv = 0; mv < moveCount; ++mv)
                for (int s = 0; s < S; ++s) out->outcomes[sample0 + (int64_t)mv * S + s] = rewards[players[mv]];
        PUT(out->game_moves, gslot, moveCount);
        PUT(out->game_samples, gslot, moveCount * S);
        PUT(out->game_rng_draws, gslot, rng.ctr);
    }
    og_free_subtree(t.game_root);
    free(players);
    free(leaves);
    return rc;
}

int oracle_selfplay_ex(const oracle_selfplay_cfg* cfg, uint64_t first_game, int ngames, oracle_selfplay_out* out,
                       oracle_search_stats* search) {
    if (!og_info(cfg->game)) return -2;
    if (cfg->evaluator == OE_CALLBACK && !cfg->eval_cb) return -2;
    out->n_moves = out->n_samples = 0;
    out->total_traversals = out->total_evals = 0;
    out->select_depth_sum = out->select_legal_sum = 0.0;
    out->select_nodes = 0;
    out->leaves_terminal = out->leaves_gray = out->leaves_empty = 0;
    if (search) memset(search, 0, sizeof(*search));
    for (int g = 0; g < ngames; ++g) {          /* selfplay/SelfPlay.hpp:203-248: games in order, concatenated */
        int rc = self_play_game(cfg, first_game + (uint64_t)g, g, out, search);
        if (rc) return rc;
    }
    return 0;
}

int oracle_selfplay(const oracle_selfplay_cfg* cfg, uint64_t first_game, int ngames, oracle_selfplay_out* out) {
    return oracle_selfplay_ex(cfg, first_game, ngames, out, NULL);
}

/* ------------------------------------------------------------------ match play */
static void match_tree_init(otree* t, const oracle_selfplay_cfg* cfg, orng_t* rng, oracle_search_stats* search) {
    memset(t, 0, sizeof(*t));
    t->cfg = cfg; t->gi = og_info(cfg->game); t->game = cfg->game; t->rng = rng; t->stats = NULL; t->search = search;
    t->game_root = og_new_root(cfg->game);
    t->game_root->own_N = &t->root_N[0];
    t->game_root->own_W = &t->root_W[0];
    t->decision = t->game_root;
}

int oracle_match_ex(const oracle_selfplay_cfg agents[2], uint64_t first_game, int ngames, oracle_match_out* out,
                    oracle_search_stats* search) {
    const ogame_info* gi = og_info(agents[0].game);
    if (!gi) return -2;
    int A = gi->actions;
    oracle_selfplay_cfg cfg[2] = { agents[0], agents[1] };
    for (int k = 0; k < 2; ++k) {               /* Evaluate.cpp:95-111; agents search with the default uWeight */
        if (cfg[k].evaluator == OE_CALLBACK && !cfg[k].eval_cb) return -2;
        cfg[k].game = agents[0].game; cfg[k].seed = agents[0].seed; cfg[k].sims = agents[0].sims;
        cfg[k].max_batch = agents[0].max_batch; cfg[k].max_queue = agents[0].max_queue;
        cfg[k].dir_eps = 0.25f; cfg[k].dir_alpha = 0.1f; cfg[k].add_noise = 1; cfg[k].u_weight = 1.0f;
    }
    out->n_moves = 0; out->wins[0] = out->wins[1] = 0; out->draws = 0;
    if (search) memset(search, 0, sizeof(*search));
    onode** leaves = (onode**)malloc(sizeof(onode*) * (size_t)(cfg[0].max_batch > 0 ? cfg[0].max_batch : 1));
    int rc = 0;
    for (int g = 0; g < ngames && rc == 0; ++g) {
        uint64_t tg = first_game + (uint64_t)g;
        orng_t rng = { cfg[0].seed, tg, 0 };
        otree tree[2];
        match_tree_init(&tree[0], &cfg[0], &rng, search);
        match_tree_init(&tree[1], &cfg[1], &rng, search);
        int moves = 0;
        while (!tree[0].decision->terminal) {   /* evaluate/play.hpp:38-57 */
            if (out->n_moves >= out->cap_moves) { rc = -1; break; }
            int player = tree[0].decision->player;
            int agent = (tg % 2 == 0) ? player : 1 - player;
            otree* t = &tree[agent];
            onode* root = t->decision;
            int traversals = 0;
            while (traversals < cfg[agent].sims) {      /* agents/UCTNetworkAgent.hpp:45-57 */
                int nleaves = 0;
                int trav = tree_search(t, leaves, &nleaves);
                if (nleaves > 0) tree_evaluate_and_backprop(t, leaves, nleaves);
                traversals += trav;
            }
            if (search) search->total_traversals += traversals;
            int64_t m = out->n_moves;
            int action = 0;                     /* std::max_element: first of the largest, :92-93 */
            for (int a = 0; a < A; ++a) {
                PUT(out->move_N, m * A + a, root->N[a]);
                PUT(out->move_W, m * A + a, root->W[a]);
                PUT(out->move_P, m * A + a, root->P[a]);
                if (root->N[a] > root->N[action]) action = a;
            }
            PUT(out->move_root_N, m, *root->own_N);
            PUT(out->move_root_W, m, *root->own_W);
            PUT(out->move_traversals, m, traversals);
            PUT(out->move_agent, m, agent);
            PUT(out->move_player, m, (int8_t)player);
            PUT(out->move_action, m, action);
            tree_advance(&tree[agent], action);         /* act(): own tree */
            tree_advance(&tree[1 - agent], action);     /* opponentAct() */
            out->n_moves += 1;
            ++moves;
        }
        if (rc == 0) {
            int winner = tree[0].decision->winner;      /* Player: -1 none */
            PUT(out->game_moves, g, moves);
            PUT(out->game_winner, g, winner);
            PUT(out->game_rng_draws, g, rng.ctr);
            if (winner == O_NONE) out->draws += 1;      /* Evaluate.cpp:141-153 */
            else out->wins[(tg % 2 == 0) ? winner : 1 - winner] += 1;
        }
        og_free_subtree(tree[0].game_root);
        og_free_subtree(tree[1].game_root);
    }
    free(leaves);
    return rc;
}

int oracle_match(const oracle_selfplay_cfg agents[2], uint64_t first_game, int ngames, oracle_match_out* out) {
    return oracle_match_ex(agents, first_game, ngames, out, NULL);
}

/* ------------------------------------------------------------------ npy I/O */
/* utils/npy.hpp:430-476: magic, v1.0, u16 LE header length, dict, pad to 16 with
 * `16 - len % 16` spaces (a full 16 when already aligned), newline, raw data. */
int oracle_write_npy_f32(const char* path, const float* data, const uint64_t* shape, int ndim) {
    char dict[256], tuple[160];
    int p = 0;
    uint64_t count = 1;
    if (ndim == 0) p += snprintf(tuple + p, sizeof(tuple) - (size_t)p, "()");
    else if (ndim == 1) p += snprintf(tuple + p, sizeof(tuple) - (size_t)p, "(%llu,)", (unsigned long long)shape[0]);
    else {
        p += snprintf(tuple + p, sizeof(tuple) - (size_t)p, "(");
        for (int i = 0; i < ndim; ++i)
            p += snprintf(tuple + p, sizeof(tuple) - (size_t)p, i + 1 < ndim ? "%llu, " : "%llu)", (unsigned long long)shape[i]);
    }
    for (int i = 0; i < ndim; ++i) count *= shape[i];
    int dl = snprintf(dict, sizeof(dict), "{'descr': '<f4', 'fortran_order': False, 'shape': %s, }", tuple);
    size_t length = 6 + 2 + 2 + (size_t)dl + 1;
    size_t pad = 16 - length % 16;
    uint16_t hlen = (uint16_t)((size_t)dl + pad + 1);
    FILE* f = fopen(path, "wb");
    if (!f) return -1;
    fwrite("\x93NUMPY\x01\x00", 1, 8, f);
    unsigned char le[2] = { (unsigned char)(hlen & 0xff), (unsigned char)(hlen >> 8) };
    fwrite(le, 1, 2, f);
    fwrite(dict, 1, (size_t)dl, f);
    for (size_t i = 0; i < pad; ++i) fputc(' ', f);
    fputc('\n', f);
    fwrite(data, sizeof(float), (size_t)count, f);
    fclose(f);
    return 0;
}

/* ------------------------------------------------------ contract unit hooks */
void oracle_dirichlet(uint64_t seed, uint64_t game, uint64_t ctr, float alpha, float* out, int n, uint64_t* ctr_out) {
    orng_t r = { seed, game, ctr };
    orng_dirichlet(&r, alpha, out, n);
    if (ctr_out) *ctr_out = r.ctr;
}
float oracle_det_powf(float x, float e) { return odet_powf(x, e); }
float oracle_det_expf(float x) { return odet_expf(x); }
uint32_t oracle_philox(uint64_t seed, uint64_t game, uint64_t ctr) { return orng_philox_word0(seed, game, ctr); }
