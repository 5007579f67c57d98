/*
 * oracle_open.c -- TEST INFRASTRUCTURE: the oracle's self-play and match play (oracle/oracle_search.c, included
 * unchanged) for games that start from opening lines.  Line i = actions[offsets[i] .. offsets[i+1]-1], a sequence of
 * actions from the start position.  Self-play game t (stream id first_game + g) starts from line t % n_lines, match game
 * t from line (t / 2) % n_lines (both colour assignments; agents[t % 2] still plays Player ZERO).  Each tree is advanced
 * through the line before its first search, as a caller of UCTTree::advanceDecision would: no random draw, the line's
 * positions are the game's history, moveCount (the temperature's counter) and every per-move output cover the searched
 * moves only.  n_lines = 0 is oracle_selfplay_ex / oracle_match_ex.  Returns -3 when a line holds an illegal action or
 * ends in a terminal position.
 *
 * open_self_play_game and oracle_match_open restate self_play_game and oracle_match_ex of the included file with the
 * opening added; everything else (search, evaluation, sampling) is the oracle's own code.  Built by
 * tests/test_openings.py together with oracle/oracle_games.c into a library of its own.
 */
#include "../oracle/oracle_search.c"

int oracle_selfplay_open(const oracle_selfplay_cfg* cfg, uint64_t first_game, int ngames, oracle_selfplay_out* out,
                         oracle_search_stats* search, int64_t n_lines, const int64_t* offsets, const int32_t* actions);
int oracle_match_open(const oracle_selfplay_cfg agents[2], uint64_t first_game, int ngames, oracle_match_out* out,
                      oracle_search_stats* search, int64_t n_lines, const int64_t* offsets, const int32_t* actions);

/* Advances a fresh tree through an opening line (uct/UCTTree.hpp:197-210).  Returns 0, or -3 when an action is not
 * legal where it is played or the line ends in a terminal position. */
static int tree_open_line(otree* t, const int32_t* line, int64_t len) {
    for (int64_t k = 0; k < len; ++k) {
        const onode* d = t->decision;
        const int a = line[k];
        if (d->terminal || a < 0 || a >= t->gi->actions || d->mask[a] == 0.0f) return -3;
        tree_advance(t, a);
    }
    return t->decision->terminal ? -3 : 0;
}

/* ------------------------------------------------------------------ selfPlay from a line */

/* selfplay/SelfPlay.hpp:50-192 for one game; appends to `out` */
static int open_self_play_game(const oracle_selfplay_cfg* cfg, uint64_t game_id, int gslot, oracle_selfplay_out* out,
                               oracle_search_stats* search, const int32_t* line, int64_t line_len) {
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
    int rc = tree_open_line(&t, line, line_len);   /* moveCount stays 0: it counts searched moves */

    while (rc == 0 && !t.decision->terminal) {
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

int oracle_selfplay_open(const oracle_selfplay_cfg* cfg, uint64_t first_game, int ngames, oracle_selfplay_out* out,
                         oracle_search_stats* search, int64_t n_lines, const int64_t* offsets, const int32_t* actions) {
    if (!og_info(cfg->game)) return -2;
    if (cfg->evaluator == OE_CALLBACK && !cfg->eval_cb) return -2;
    out->n_moves = out->n_samples = 0;
    out->total_traversals = out->total_evals = 0;
    out->select_depth_sum = out->select_legal_sum = 0.0;
    out->select_nodes = 0;
    out->leaves_terminal = out->leaves_gray = out->leaves_empty = 0;
    if (search) memset(search, 0, sizeof(*search));
    for (int g = 0; g < ngames; ++g) {          /* selfplay/SelfPlay.hpp:203-248: games in order, concatenated */
        const uint64_t id = first_game + (uint64_t)g;
        const int64_t li = n_lines > 0 ? (int64_t)(id % (uint64_t)n_lines) : 0;
        int rc = n_lines > 0 ? open_self_play_game(cfg, id, g, out, search, actions + offsets[li], offsets[li + 1] - offsets[li])
                             : open_self_play_game(cfg, id, g, out, search, NULL, 0);
        if (rc) return rc;
    }
    return 0;
}

/* ------------------------------------------------------------------ match play */
int oracle_match_open(const oracle_selfplay_cfg agents[2], uint64_t first_game, int ngames, oracle_match_out* out,
                      oracle_search_stats* search, int64_t n_lines, const int64_t* offsets, const int32_t* actions) {
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
        if (n_lines > 0) {                      /* ids 2k and 2k+1 play one line with the colours swapped */
            const int64_t li = (int64_t)((tg / 2) % (uint64_t)n_lines);
            const int64_t len = offsets[li + 1] - offsets[li];
            rc = tree_open_line(&tree[0], actions + offsets[li], len);
            if (rc == 0) rc = tree_open_line(&tree[1], actions + offsets[li], len);
        }
        int moves = 0;
        while (rc == 0 && !tree[0].decision->terminal) {   /* evaluate/play.hpp:38-57 */
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
