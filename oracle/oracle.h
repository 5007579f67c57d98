/*
 * oracle.h -- TEST INFRASTRUCTURE.  Plain-C restatement of the reference's
 * self-play hot path (willwin4sure/sprl, cpp/src).  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load this library; the product (sprl_b200/) never does.
 *
 * Parity status: PINNED.  Every function here is checked against the
 * reference's own sources compiled verbatim (oracle/_ref/ref_trace, built by
 * oracle/Makefile from /root/reference/cpp/src) through the golden fixtures in
 * tests/golden/ (generator: tests/golden/make_golden.py) and against the one
 * known-answer test the reference holds (cpp/tests/test_c4.cpp:5-25).
 *
 * Citations "games/..", "uct/..", "selfplay/..", "symmetry/..", "networks/..",
 * "utils/.." are relative to /root/reference/cpp/src/.
 */
#ifndef SPRL_ORACLE_H
#define SPRL_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { OG_OTHELLO = 0, OG_C4 = 1, OG_GO7 = 2, OG_GO9 = 3 };
enum { OE_UNIFORM = 0, OE_HASHNET = 1, OE_CALLBACK = 2, OE_HEURISTIC = 3 /* networks/OthelloHeuristic.cpp, Othello only */ };
enum { OQ_ZERO = 0, OQ_PARENT = 1, OQ_DROP_PARENT = 2 };

#define OG_MAXB 81
#define OG_MAXA 82
#define OG_MAXH 8

typedef struct {
    int rows, cols, cells, actions, history, nsym, max_plies;
    float komi;
} ogame_info;

int oracle_game_info(int game, ogame_info* out);

/* Leaf-count perft from the start position: a pass is a ply, a terminal node
 * above the horizon counts 1. */
int oracle_perft(int game, int depth, uint64_t* count);

/* Random playouts: the move is legal[UniformInt(0, nlegal-1)] from the contract
 * stream (seed, first_game + g).  Every visited position (start and terminal
 * included) is recorded.  Returns the number of positions, or -1 when `cap`
 * positions do not suffice. */
int64_t oracle_rollout(int game, uint64_t seed, uint64_t first_game, int ngames, int64_t cap,
                       int32_t* game_steps, int8_t* cells, int8_t* player, int8_t* terminal,
                       int8_t* winner, int8_t* mask, int32_t* action);

/* Replay a fixed action list from the start position (known-answer tests). */
int oracle_replay(int game, const int32_t* actions, int n, int8_t* cells, int8_t* player,
                  int8_t* terminal, int8_t* winner, int8_t* mask, float* rewards2);

/* Evaluator callback: planes [n, 2H+1, R, C] fp32 -> logits [n, A], values [n]. */
typedef void (*oracle_eval_cb)(void* user, const float* planes, int n, float* logits, float* values);

typedef struct {
    int game;
    int evaluator;      /* OE_* */
    uint64_t seed;
    int sims;           /* numTraversals per move */
    int max_batch;
    int max_queue;
    float dir_eps;
    float dir_alpha;
    int add_noise;
    int use_sym;
    int init_q;         /* OQ_* */
    float u_weight;     /* constants.hpp:6 U_WEIGHT = 1.1f */
    oracle_eval_cb eval_cb;
    void* eval_user;
    uint64_t hash_salt; /* OE_HASHNET: 0 = the plain net, other values = independent nets (matches) */
    int fix_symmetry_mask; /* NOT the reference: symmetrise the legal mask together with the state before the
                            * evaluator masks its policy (repairs quirk Q3, uct/UCTTree.hpp:136-149).  Default 0. */
    int caller_moves;      /* 1: the tree is driven through UCTTree's public API by a caller that plays the FIRST
                            * most-visited action (ref_trace `treewalk`): no SampleCDF draw, advanceDecision(argmax). */
} oracle_selfplay_cfg;

typedef struct {
    /* capacities supplied by the caller */
    int64_t cap_moves, cap_samples;
    /* per game [ngames] */
    int32_t* game_moves;
    int32_t* game_samples;
    uint64_t* game_rng_draws;
    /* per move [cap_moves (x A | x B)] */
    float* move_N;
    float* move_W;
    float* move_P;
    float* move_root_N;
    float* move_root_W;
    int32_t* move_action;
    int32_t* move_traversals;
    int32_t* move_evals;
    int8_t* move_player;
    int8_t* move_board;
    /* samples [cap_samples ...] in the layout of selfplay/GridWorker.hpp:146-196 */
    float* states;         /* [S, 2H+1, R, C] */
    float* distributions;  /* [S, A] */
    float* outcomes;       /* [S] */
    /* totals written back */
    int64_t n_moves, n_samples;
    int64_t total_traversals, total_evals;
    double select_depth_sum;   /* sum over descents of nodes on the path below the root */
    double select_legal_sum;   /* sum over expanded nodes visited of their legal-child count */
    int64_t select_nodes;      /* expanded nodes visited during descents */
    int64_t leaves_terminal, leaves_gray, leaves_empty;
} oracle_selfplay_out;

/* selfPlay + runIteration (selfplay/SelfPlay.hpp:50-248) for games
 * first_game .. first_game+ngames-1, each on its own contract stream.
 * Any output pointer may be NULL.  Returns 0, or -1 on capacity overflow. */
int oracle_selfplay(const oracle_selfplay_cfg* cfg, uint64_t first_game, int ngames,
                    oracle_selfplay_out* out);

/* Match play between two evaluators (Evaluate.cpp:93-157: UCTNetworkAgent::act, agents/UCTNetworkAgent.hpp:42-108,
 * inside playGame, evaluate/play.hpp:24-69).  Each side owns a tree (Dirichlet noise on, eps 0.25, alpha 0.1, default
 * uWeight 1.0) and its own evaluator / symmetrizer / init-Q (`agents[k]`: evaluator, hash_salt, use_sym, init_q, eval_cb
 * are read from it; game, seed, sims, max_batch, max_queue from agents[0]).  Game t = first_game + g: agents[t % 2]
 * plays Player ZERO.  The mover searches `sims` descents, plays the FIRST action with the most visits, and both trees
 * advance.  Per-move arrays describe the mover's root. */
typedef struct {
    int64_t cap_moves;
    int32_t* game_moves;      /* [ngames] */
    int32_t* game_winner;     /* [ngames] -1 none / 0 / 1 (Player) */
    uint64_t* game_rng_draws; /* [ngames] */
    float* move_N; float* move_W; float* move_P;   /* [cap_moves, A] */
    float* move_root_N; float* move_root_W;        /* [cap_moves] */
    int32_t* move_action; int32_t* move_traversals; int32_t* move_agent;
    int8_t* move_player;
    int64_t n_moves;
    int64_t wins[2];          /* games won by agents[0] / agents[1] */
    int64_t draws;
} oracle_match_out;

int oracle_match(const oracle_selfplay_cfg agents[2], uint64_t first_game, int ngames, oracle_match_out* out);

/* Shape of the searches (counters only: they change no other output).  A descent's depth is the number of edges
 * chosen below the decision node.  The search kernel records up to 32 edges of a descent for its parallel backup and
 * backs deeper ones up by parent links; its leaf-batch deduplication compares the first 32 queue entries only.
 * A separate struct, filled by the _ex entry points, so that callers of the structs above keep their layout. */
#define ODEPTH_BINS 128
typedef struct {
    int64_t total_traversals, total_evals;
    int64_t leaves_terminal, leaves_gray, leaves_empty;
    double select_depth_sum, select_legal_sum;
    int32_t select_depth_max;
    int64_t depth_hist[ODEPTH_BINS];    /* descents by depth, the last bin counts every depth >= 127 */
    int64_t deep_terminal, deep_gray, deep_queued;   /* descents of >= 32 edges by how their leaf was handled */
    int32_t queue_max;                  /* most leaves queued by one searchAndGetLeaves call */
    int64_t dup_total;                  /* queued leaves already queued earlier in the same batch */
    int64_t dup_first32;                /* the same, counted only among the first 32 entries of each batch */
} oracle_search_stats;

/* oracle_selfplay / oracle_match that also fill `search` (may be NULL); in a match it sums both agents' searches. */
int oracle_selfplay_ex(const oracle_selfplay_cfg* cfg, uint64_t first_game, int ngames, oracle_selfplay_out* out,
                       oracle_search_stats* search);
int oracle_match_ex(const oracle_selfplay_cfg agents[2], uint64_t first_game, int ngames, oracle_match_out* out,
                    oracle_search_stats* search);

/* .npy v1.0 writer restated from utils/npy.hpp:430-476,616-639 (float32, C order). */
int oracle_write_npy_f32(const char* path, const float* data, const uint64_t* shape, int ndim);

/* Exposed pieces of the contract for unit tests. */
void oracle_dirichlet(uint64_t seed, uint64_t game, uint64_t ctr, float alpha, float* out, int n, uint64_t* ctr_out);
float oracle_det_powf(float x, float e);
float oracle_det_expf(float x);
uint32_t oracle_philox(uint64_t seed, uint64_t game, uint64_t ctr);
void oracle_symmetrize_cells(int game, int sym, const int8_t* in, int8_t* out);
void oracle_symmetrize_dist(int game, int sym, const float* in, float* out);
int oracle_inverse_symmetry(int game, int sym);
void oracle_hashnet(int game, const int8_t* hist_cells, int hist_size, int player, const float* mask,
                    float* policy, float* value);

#ifdef __cplusplus
}
#endif
#endif
