/*
 * sprl_b200.h -- C ABI of libsprl_b200.so, the B200-native self-play engine.
 *
 * The reference (willwin4sure/sprl) has no FFI: its hot path is a C++ template
 * library (cpp/src/{games,uct,networks,symmetry,selfplay}) driven by
 * cpp/src/OTHWorker.cpp.  This header is the boundary a maintainer binds
 * instead of instantiating those templates; each entry point names the
 * reference interface it replaces (paths relative to /root/reference/cpp/src).
 *
 * Conventions: plain pointers and sizes, no C++ or torch types.  Every function
 * returns 0 on success or a negative SPRL_E_* code; sprl_last_error() gives the
 * message of the last failure on the calling thread.  Pointers named h_* are
 * host memory, d_* device memory of the engine's GPU.  An engine handle is not
 * thread-safe; use one host thread per engine (= per GPU).
 */
#ifndef SPRL_B200_H
#define SPRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPRL_OK 0
#define SPRL_E_INVALID (-1)    /* bad argument */
#define SPRL_E_CUDA (-2)       /* CUDA runtime error (sticky on the engine) */
#define SPRL_E_CAPACITY (-3)   /* a caller buffer or a device pool is too small */
#define SPRL_E_STATE (-4)      /* call not valid in the engine's current state */
#define SPRL_E_IO (-5)         /* file could not be written */
#define SPRL_E_NOGPU (-6)      /* no CUDA device: there is no CPU fallback */

/* games/{OthelloNode,ConnectFourNode,GoNode}.hpp */
#define SPRL_GAME_OTHELLO 0
#define SPRL_GAME_C4 1
#define SPRL_GAME_GO7 2
#define SPRL_GAME_GO9 3

/* networks/INetwork.hpp implementations */
#define SPRL_EVAL_UNIFORM 0    /* networks/RandomNetwork.hpp:21-49, evaluated on device */
#define SPRL_EVAL_HASHNET 1    /* deterministic test evaluator, evaluated on device */
#define SPRL_EVAL_EXTERNAL 2   /* networks/GridNetwork.hpp:62-145: caller runs the traced network on device buffers */
#define SPRL_EVAL_OTHELLO_HEURISTIC 3 /* networks/OthelloHeuristic.cpp:5-53 (Othello only), evaluated on device */

/* uct/UCTNode.hpp:24-28 */
#define SPRL_INITQ_ZERO 0
#define SPRL_INITQ_PARENT 1
#define SPRL_INITQ_DROP_PARENT 2 /* :152-163,196-206: unvisited children answer with the node's own Q = W/N */

const char* sprl_last_error(void);
int sprl_device_count(void);

typedef struct {
    int rows, cols, cells, actions, history, nsym, max_plies;
} sprl_game_info;

/* Compile-time constants of a game (games/OthelloNode.hpp:8-11 etc.). */
int sprl_game_info_get(int game, sprl_game_info* out);

/* ------------------------------------------------------------------ environment
 * Batched rules without a tree: replaces GameNode::getAddChild / getActionMask /
 * isTerminal / getWinner (games/GameNode.hpp:96-160) over many positions. */

/* One transition per position.  Inputs (host): cells [n, cells] int8 with the
 * reference's Piece encoding (-1 empty, 0, 1), player [n] (0/1), action [n].
 * Outputs (host): next cells, next player, terminal, winner (-1/0/1), mask
 * [n, actions] (0/1).  Othello and Connect Four only (Go needs the history path:
 * use sprl_env_rollout / sprl_env_perft). */
int sprl_env_step(int device, int game, int64_t n, const int8_t* h_cells, const int8_t* h_player,
                  const int32_t* h_action, int8_t* h_next_cells, int8_t* h_next_player,
                  int8_t* h_terminal, int8_t* h_winner, int8_t* h_mask);

/* One line of play from the start position: h_actions[0 .. n_actions-1] in order -- the chain of
 * GameNode::getAddChild calls of a host program (games/GameNode.hpp:96-110; the start position is the node
 * constructor's setStartNode, :176), for every game incl. Go (the line itself is the history of the positional-superko
 * rule, games/GoNode.cpp:88-170).  Outputs (host, any may be NULL) for the n_actions + 1 positions along the line, start
 * position first: cells [n+1, cells], player / terminal / winner [n+1], mask [n+1, actions], encodings as in
 * sprl_env_step.  An action that is not legal where it is played fails with SPRL_E_INVALID (the reference asserts). */
int sprl_env_line(int device, int game, int32_t n_actions, const int32_t* h_actions, int8_t* h_cells, int8_t* h_player,
                  int8_t* h_terminal, int8_t* h_winner, int8_t* h_mask);

/* Random playouts from the start position, one GPU thread per game; move k of
 * game g is legal[UniformInt(0, nlegal-1)] from the stream (seed, first_game+g).
 * h_game_steps [ngames] receives positions per game (start and terminal
 * included), h_final_winner [ngames] the winner.  When h_cells != NULL every
 * position is recorded in playing order (game-major), up to `cap` positions:
 * cells [cap, cells], player/terminal/winner [cap], mask [cap, actions],
 * action [cap] (-1 at terminal positions).  total_positions receives the count.
 * elapsed_ms (optional) receives the device time of the playout kernel alone. */
int sprl_env_rollout(int device, int game, uint64_t seed, uint64_t first_game, int64_t ngames,
                     int32_t* h_game_steps, int8_t* h_final_winner, int64_t cap,
                     int8_t* h_cells, int8_t* h_player, int8_t* h_terminal, int8_t* h_winner,
                     int8_t* h_mask, int32_t* h_action, int64_t* total_positions, float* elapsed_ms);

/* Leaf-count perft from the start position by breadth-first frontier expansion
 * on the device (a pass is a ply; a terminal node above the horizon counts 1). */
int sprl_env_perft(int device, int game, int depth, uint64_t* count, float* elapsed_ms);

/* ------------------------------------------------------------------ self-play engine
 * Replaces UCTTree (uct/UCTTree.hpp:38-210), selfPlay / runIteration
 * (selfplay/SelfPlay.hpp:50-248) and the sample embedding + .npy dump of runWorker
 * (selfplay/GridWorker.hpp:143-196) for `num_slots` concurrent games on one GPU. */
typedef struct sprl_engine sprl_engine;

typedef struct {
    int device;             /* CUDA device ordinal */
    int game;               /* SPRL_GAME_* */
    int evaluator;          /* SPRL_EVAL_* */
    uint64_t seed;          /* run seed of the counter-based streams (constants.hpp:4 SEED) */
    int num_slots;          /* concurrent games (trees) on the device */
    int sims;               /* numTraversals per move (OTHWorker.cpp:23 UCT_TRAVERSALS) */
    int max_batch;          /* maxBatchSize (OTHWorker.cpp:24) */
    int max_queue;          /* maxQueueSize (OTHWorker.cpp:25) */
    float dir_eps;          /* OTHWorker.cpp:27 */
    float dir_alpha;        /* OTHWorker.cpp:28 */
    float u_weight;         /* constants.hpp:6 U_WEIGHT */
    int add_noise;          /* Dirichlet noise at the decision node */
    int use_sym;            /* symmetrizer present: random symmetry per leaf, S-fold samples */
    int init_q;             /* SPRL_INITQ_* (GridWorker.hpp:141 uses PARENT) */
    int64_t units_per_tree; /* 16-byte units per tree slab; 0 = derive from sims */
    int64_t max_games;      /* capacity of the per-game records (games per iteration) */
    int record_stats;       /* keep per-move root N/W/P for sprl_move_stats (parity tests) */
    int rounds_per_launch;  /* device evaluators: search rounds per kernel launch; 0 = default */
    int fix_symmetry_mask;  /* 0 = the reference (quirk: the evaluator masks a symmetrised policy with the UN-symmetrised
                             * legal mask, uct/UCTTree.hpp:136-149, networks/GridNetwork.hpp:117-125, so legal moves can get
                             * prior 0); 1 = the mask is symmetrised with the state.  Not the reference's behaviour. */
} sprl_config;

/* Fills a config with the reference's Othello worker constants (OTHWorker.cpp:12-28,
 * constants.hpp) for `game`; the caller then overrides what it needs. */
int sprl_default_config(int game, sprl_config* cfg);

int sprl_create(const sprl_config* cfg, sprl_engine** out);
void sprl_destroy(sprl_engine* e);

/* All engine work is enqueued on this CUDA stream (a cudaStream_t; NULL = default). */
int sprl_set_stream(sprl_engine* e, void* cuda_stream);

/* SPRL_EVAL_EXTERNAL: device buffers of the traced network's input and outputs
 * (networks/GridNetwork.hpp:70,99-102), capacity batch = num_slots * max_queue rows:
 * d_in [batch, 2H+1, R, C] is WRITTEN by sprl_round; d_logits [batch, A] and d_value [batch]
 * are READ by the next sprl_round.  A launch hands out rows compactly, in no particular
 * order, to the leaves it queued: only rows [0, d_rows[0]) hold leaves (sprl_eval_rows), the
 * others keep stale data and their outputs are never read. */
int sprl_bind_eval_buffers(sprl_engine* e, float* d_in, const float* d_logits, const float* d_value);
int64_t sprl_eval_batch(const sprl_engine* e);
/* Device address of the row counts of the last launch (uint32_t[2], updated on the stream by every
 * sprl_round): d_rows[0] rows from row 0 hold leaves; in match play d_rows[0] counts agent 0's rows
 * [0, d_rows[0]) and d_rows[1] agent 1's rows [half, half + d_rows[1]).  An evaluator that can read its
 * batch size on the device (sprl_evalnet_forward_counted) skips the rest. */
int sprl_eval_rows(sprl_engine* e, const uint32_t** d_rows);

/* Starts runIteration(num_games): games first_game .. first_game+num_games-1, game g on
 * stream (seed, g), slot s plays games s, s+num_slots, ... one after the other. */
int sprl_begin_iteration(sprl_engine* e, uint64_t first_game, int64_t num_games);

/* Sharding across GPUs (one engine per rank): game i of an iteration uses stream id
 * first_game + i * stride, so rank r of `world` plays ids r, r+world, ... with
 * first_game = base + r and stride = world.  Default stride 1. */
int sprl_set_game_stride(sprl_engine* e, uint64_t stride);

/* Opening lines for the games / trees the NEXT sprl_begin_iteration, sprl_match_begin or sprl_begin_trees starts.
 * Line i = h_actions[h_offsets[i] .. h_offsets[i+1]-1], a sequence of actions from the start position; n_lines = 0
 * turns openings off (the default).  Self-play games and step-wise trees with stream id t start from line t % n_lines;
 * match games from line (t / 2) % n_lines, so that ids 2k and 2k+1 play one line with the colours swapped (agent t % 2
 * still plays Player ZERO).  Starting from a line means exactly: the tree is built at the start position and advanced
 * through the line (as sprl_advance does) before any search.  The line draws no random numbers, its positions are the
 * game's history (network inputs, sample planes, Go's superko), and the decision node starts unsearched.  Samples, move
 * statistics, move counts (sprl_iteration_counts, sprl_move_stats, sprl_match_results, sprl_stats.moves) cover the
 * searched moves only; the temperature of self-play counts searched moves; the outcome is that of the finished game.
 * Every line is replayed once on the device when it is set.  Fails with SPRL_E_INVALID for an illegal action or a line
 * that reaches a terminal position (message names line and ply), SPRL_E_STATE while an iteration / match / set of
 * trees is open (still has a game or tree playing); the previous lines then stay in force. */
int sprl_set_openings(sprl_engine* e, int64_t n_lines, const int64_t* h_offsets, const int32_t* h_actions);

/* Enqueues one search launch: apply the evaluations of the previous launch, finish
 * moves whose traversal budget is spent (sample, re-root, compact), then run the next
 * searchAndGetLeaves batch of every live tree.  Asynchronous, capturable in a CUDA graph. */
int sprl_round(sprl_engine* e);

/* Synchronises the stream; reports slots still playing and slots stopped by an error. */
int sprl_poll(sprl_engine* e, int64_t* slots_playing, int64_t* slots_failed);

/* Evaluator callback for sprl_run_iteration with SPRL_EVAL_EXTERNAL: run the network
 * on d_in (batch rows) and leave its outputs in d_logits / d_value, on `cuda_stream`. */
typedef int (*sprl_forward_fn)(void* user, const float* d_in, int64_t batch, float* d_logits, float* d_value,
                               void* cuda_stream);

/* begin + rounds until every game is finished.  forward may be NULL for device evaluators. */
int sprl_run_iteration(sprl_engine* e, uint64_t first_game, int64_t num_games, sprl_forward_fn forward, void* user);

/* Totals of the finished iteration. */
int sprl_iteration_counts(sprl_engine* e, int64_t* n_moves, int64_t* n_samples);

/* Writes the iteration's samples, in the reference's order (games, moves, symmetries),
 * to HOST arrays: states [n, 2H+1, R, C], distributions [n, A], outcomes [n]. */
int sprl_collect_samples(sprl_engine* e, int64_t cap_samples, float* h_states, float* h_distributions,
                         float* h_outcomes, int64_t* n_samples);
/* Streamed output: registers the HOST arrays the next iterations' samples go to (same layout and order as
 * sprl_collect_samples; capacity cap_samples rows).  From then on every sprl_poll embeds the games that have finished
 * -- in game order, a game's rows follow those of all earlier games -- and copies them on a side stream while the other
 * games keep playing, and sprl_collect_samples called with the SAME three pointers only waits for the rest.  pin != 0
 * page-locks the arrays (cudaHostRegister) for the lifetime of the registration: asynchronous, full-speed copies.
 * Three NULL pointers turn streaming off.  The arrays must stay valid until then or until sprl_destroy. */
int sprl_stream_samples(sprl_engine* e, int64_t cap_samples, float* h_states, float* h_distributions, float* h_outcomes, int pin);
/* Progress of the streamed output: games and sample rows copied so far in the open iteration, and (since the
 * registration) how many chunks left while games were still being played. */
int sprl_stream_info(sprl_engine* e, int64_t* games_done, int64_t* samples_done, uint64_t* chunks_while_playing);
/* Same, left on the device (engine-owned, valid until the next begin/collect). */
int sprl_collect_samples_device(sprl_engine* e, float** d_states, float** d_distributions, float** d_outcomes,
                                int64_t* n_samples);

/* Per-move search record of the iteration (needs record_stats), move-major in game order:
 * N, W, P [n_moves, A]; root_N, root_W [n_moves]; action, traversals [n_moves];
 * player [n_moves]; game_moves [num_games]; game_draws [num_games] (RNG draws used). */
int sprl_move_stats(sprl_engine* e, int64_t cap_moves, float* h_N, float* h_W, float* h_P, float* h_root_N,
                    float* h_root_W, int32_t* h_action, int32_t* h_traversals, int8_t* h_player,
                    int32_t* h_game_moves, uint64_t* h_game_draws, int64_t* n_moves);

/* ------------------------------------------------------------------ match play
 * Replaces Evaluate.cpp:93-157: UCTNetworkAgent::act / opponentAct (agents/UCTNetworkAgent.hpp:42-108) inside
 * playGame (evaluate/play.hpp:24-69), for num_slots / 2 concurrent games.  Each game is served by two trees, one
 * per side, with its own evaluator, symmetrizer and init-Q; the side to move spends `sims` descents in its tree,
 * plays the first action with the most visits, and both trees advance.  Game t (stream id, as in self-play) gives
 * Player ZERO to agent t % 2.  Search constants come from the engine's config (Evaluate.cpp uses Dirichlet noise
 * on, eps 0.25, alpha 0.1 and the default uWeight 1.0).  Trees [0, num_slots/2) belong to agent 0 and
 * [num_slots/2, 2 * (num_slots/2)) to agent 1, so with SPRL_EVAL_EXTERNAL the first half of the evaluator batch
 * (row tree * max_queue + q) is agent 0's network input and the second half agent 1's. */
typedef struct {
    int evaluator;          /* SPRL_EVAL_* of this side */
    int use_sym;            /* Evaluate.cpp model<k>UseSymmetrize */
    int init_q;             /* Evaluate.cpp model<k>UseParentQ ? PARENT : ZERO */
    uint64_t hash_salt;     /* SPRL_EVAL_HASHNET: 0 = the plain test net, other values = independent nets */
} sprl_agent_config;

/* Starts a match of games first_game .. (stride as in self-play); then sprl_round / sprl_poll as usual. */
int sprl_match_begin(sprl_engine* e, const sprl_agent_config* h_agents /* [2] */, uint64_t first_game, int64_t num_games);

/* begin + rounds until every game is finished.  With SPRL_EVAL_EXTERNAL agents `forward` is called once per round
 * for the WHOLE batch; it runs agent 0's network on rows [0, half) and agent 1's on [half, 2*half),
 * half = (num_slots / 2) * max_queue (skipping a side that uses a device evaluator). */
int sprl_run_match(sprl_engine* e, const sprl_agent_config* h_agents /* [2] */, uint64_t first_game, int64_t num_games,
                   sprl_forward_fn forward, void* user);

/* Results of the finished match: per game the winner (-1 none / 0 / 1 = Player), moves played and RNG draws used
 * (any of them may be NULL); wins[2] = games won by agent 0 / agent 1, draws (Evaluate.cpp:139-155). */
int sprl_match_results(sprl_engine* e, int64_t cap_games, int8_t* h_winner, int32_t* h_moves, uint64_t* h_draws,
                       int64_t* wins /* [2] */, int64_t* draws);

/* ------------------------------------------------------------------ step-wise trees
 * UCTTree's public surface (uct/UCTTree.hpp:38-210) for many independent trees at once: what the move loops of
 * selfPlay (selfplay/SelfPlay.hpp:82-146) and UCTNetworkAgent::act / opponentAct (agents/UCTNetworkAgent.hpp:42-108)
 * do by hand -- search some descents, read the decision node's statistics, advance by an action of the CALLER's
 * choice.  Search constants, evaluator, symmetrizer, noise and init-Q come from the engine's config. */

/* UCTTree(root = start position, ...) (uct/UCTTree.hpp:38-57) for trees 0 .. num_trees-1 (<= num_slots); tree i draws
 * from stream first_game + i * stride, as game i of an iteration would. */
int sprl_begin_trees(sprl_engine* e, uint64_t first_game, int64_t num_trees);
/* while (traversals < sims) { searchAndGetLeaves(maxBatch, maxQueue); evaluateAndBackpropLeaves(leaves); } for every
 * live tree (uct/UCTTree.hpp:76-184 as driven by selfplay/SelfPlay.hpp:100-108; the loop adds whole batches, so a tree
 * ends with sims .. sims + max_batch - 1 descents since its last advance).  Returns when every tree has spent its
 * budget and all evaluations are backed up.  forward: as in sprl_run_iteration (NULL for device evaluators). */
int sprl_search(sprl_engine* e, int sims, sprl_forward_fn forward, void* user);
/* The two halves of one such loop trip, for callers that drive the evaluator themselves (a CUDA graph, another
 * stream): sprl_search_batch enqueues ONE searchAndGetLeaves batch per live tree (leaf planes -> d_in, row counts ->
 * sprl_eval_rows); after the network has written d_logits / d_value, sprl_apply_evaluations enqueues
 * evaluateAndBackpropLeaves (:124-184) for the queued leaves.  Both asynchronous on the engine's stream. */
int sprl_search_batch(sprl_engine* e);
int sprl_apply_evaluations(sprl_engine* e);
/* getDecisionNode() (uct/UCTTree.hpp:62) of every tree: its EdgeStatistics (uct/UCTNode.hpp:45-60) as dense rows
 * N, W, P [num_trees, A] (P = the child priors in use: Dirichlet-mixed when add_noise; 0 before the node is expanded),
 * the node's own N / W (the tree-level edge, uct/UCTTree.hpp:301), player to move, terminal flag, winner (-1/0/1),
 * descents since the last advance, the legal mask [num_trees, A] (GameNode::getActionMask) and the number of leaves
 * queued for the evaluator (what the last searchAndGetLeaves returned).  Host arrays; any may be NULL.  Synchronises
 * the stream. */
int sprl_root_stats(sprl_engine* e, int64_t cap_trees, float* h_N, float* h_W, float* h_P, float* h_root_N, float* h_root_W,
                    int8_t* h_player, int8_t* h_terminal, int8_t* h_winner, int32_t* h_traversals, int8_t* h_mask,
                    int32_t* h_queued);
/* advanceDecision(h_actions[i]) for tree i (uct/UCTTree.hpp:197-210: prune the siblings, clear the kept subtree's
 * statistics, keep its cached evaluations); -1 leaves a tree where it is.  An illegal action fails with
 * SPRL_E_INVALID.  A tree whose new decision node is terminal stops (sprl_poll counts it as finished). */
int sprl_advance(sprl_engine* e, const int32_t* h_actions, int64_t n_actions);

typedef struct {
    uint64_t sims, evals, moves, games;
    uint64_t depth_sum, legal_sum, nodes_visited;
    uint64_t leaves_terminal, leaves_gray, leaves_empty;
    uint64_t units_high_water;      /* largest slab fill seen by any tree */
    uint64_t units_per_tree;
    uint64_t launches;              /* kernels this engine launched since creation */
    uint64_t device_bytes;          /* HBM held by the engine */
    uint64_t leaves_duplicate;      /* queued leaves that were already queued in the same batch (uct/UCTTree.hpp:166-182:
                                     * evaluated again by the reference, result dropped): counted in `evals` like the
                                     * reference's getNumEvals, but they take no evaluator row -- rows = evals - this */
} sprl_stats;

/* Counters accumulated since sprl_create (or the last sprl_reset_stats). */
int sprl_get_stats(sprl_engine* e, sprl_stats* out);
int sprl_reset_stats(sprl_engine* e);

/* Debug aid (the reference has no race or bounds tooling, SURVEY.md section 5): every device pool of the engine lies
 * between two 256-byte guard bands; this synchronises the device and reports how many pools have a damaged band,
 * i.e. were written out of bounds by a kernel. */
int sprl_debug_check_guards(sprl_engine* e, int64_t* pools_checked, int64_t* pools_damaged);

/* npy::write_npy (utils/npy.hpp:616-639) for float32 C-order data: byte-identical header. */
int sprl_write_npy_f32(const char* path, const float* h_data, const uint64_t* shape, int ndim);

/* ------------------------------------------------------------------ evaluator network
 * The forward pass of the controller's network (src/networks/grid_networks.py:30-80
 * BasicGridNetwork, loaded by networks/GridNetwork.hpp:37-51 and run at :99) as one persistent
 * tcgen05 kernel for boards up to 8x8 (Othello, Go 7x7, Connect Four: two boards per MMA tile) and up
 * to 128 cells in rows of at most 16 (Go 9x9: one board per tile): conv tower on the tensor cores with
 * a two-term fp16 split (fp32-level accuracy, fp32 accumulate), BatchNorm folded, head FCs in a second
 * kernel.  Limits: 1 to 21 input planes, 0 to 7 residual blocks of 64 or 128 channels, a value hidden layer as
 * wide as the tower, 1 or 2 policy channels, 1 to 84 actions.  The head FCs stage their weights and a step of head
 * activations in shared memory: with 64 channels a 64-board step, which caps boards with two policy channels at
 * 87 cells (Go 9x9's 81 fit); with 128 channels a 32-board step, which caps them at 110 cells.  With one policy
 * channel the whole 128 cells fit at both widths.  128-channel networks always run the streaming kernel (one CTA
 * per SM; a layer's weights do not fit the resident kernel), so for them SPRL_EVALNET_PATH_RESIDENT and
 * SPRL_EVALNET_PRECISION_FP16 fail with SPRL_E_STATE.  Other shapes keep using the traced module through
 * sprl_forward_fn. */
typedef struct {
    const float *weight, *bias;                             /* conv: [out, in, 3, 3], [out] */
    const float *bn_weight, *bn_bias, *bn_mean, *bn_var;    /* BatchNorm2d affine + running stats, [out] */
} sprl_conv_bn_params;

typedef struct {
    int rows, cols, in_planes, channels, blocks, actions;   /* BasicGridNetwork(rows, cols, actions, (in_planes-1)/2, blocks, channels) */
    int policy_channels, value_channels, value_hidden;      /* 2, 1, channels */
    float bn_eps;                                           /* 0 = 1e-5 */
    sprl_conv_bn_params stem;                               /* conv, bn */
    const sprl_conv_bn_params* tower;                       /* [2 * blocks]: conv1/bn1, conv2/bn2 of every residual block */
    const float *policy_conv_w, *policy_conv_b;             /* [policy_channels, channels, 1, 1], [policy_channels] */
    const float *policy_fc_w, *policy_fc_b;                 /* [actions, policy_channels * rows * cols], [actions] */
    const float *value_conv_w, *value_conv_b;               /* [1, channels, 1, 1], [1] */
    const float *value_fc1_w, *value_fc1_b;                 /* [value_hidden, rows * cols], [value_hidden] */
    const float *value_fc2_w, *value_fc2_b;                 /* [1, value_hidden], [1] */
} sprl_network_params;                                      /* all pointers are HOST memory */

typedef struct sprl_evalnet sprl_evalnet;

int sprl_evalnet_create(int device, const sprl_network_params* h_params, sprl_evalnet** out);
/* New generation's weights, same shape (a change of width is refused): overwritten in place.  Device addresses stay valid, and the per-layer
 * weight scales live in device memory too, so a CUDA graph captured before the update replays with the new
 * weights and their scales. */
int sprl_evalnet_update(sprl_evalnet* net, const sprl_network_params* h_params);
/* INetwork::evaluate's forward (networks/GridNetwork.hpp:99-102) on device buffers:
 * d_in [batch, in_planes, rows, cols] -> d_logits [batch, actions], d_value [batch].  Asynchronous on
 * `cuda_stream`; matches sprl_forward_fn so that it can serve as the engine's evaluator. */
int sprl_evalnet_forward(sprl_evalnet* net, const float* d_in, int64_t batch, float* d_logits, float* d_value,
                         void* cuda_stream);
/* Same with the batch size read on the device at run time: rows [0, min(*d_rows, max_batch)) are evaluated.
 * The launch is sized for max_batch, so it can sit in a CUDA graph while the leaf count changes every round. */
int sprl_evalnet_forward_counted(sprl_evalnet* net, const float* d_in, const uint32_t* d_rows, int64_t max_batch,
                                 float* d_logits, float* d_value, void* cuda_stream);
/* Synchronises the device and reports a kernel-side failure, if any. */
int sprl_evalnet_status(sprl_evalnet* net, uint64_t* launches);
/* Bytes copied host -> device by one create / update, weight-ring depth and shared memory per CTA. */
int sprl_evalnet_info(sprl_evalnet* net, int64_t* upload_bytes, int32_t* ring_stages, int32_t* smem_bytes);
/* Which kernel runs the conv tower.  AUTO: the resident-weight kernel (csrc/evalnet_resident.cuh: the weights of one
 * residual block stay in shared memory for a whole launch, one launch per block; boards of up to 128 cells incl. Go 9x9)
 * when a block fits, else the streaming kernel (weights re-read from L2 per tile).  Both accumulate the conv tower in
 * the same order; the resident kernel computes the 1x1 head convolutions as fp32 FMAs instead of split-fp16 MMAs, so
 * their outputs agree to rounding (1e-6), each within 2e-6 of the fp64 forward.  STREAMING / RESIDENT force one of
 * them (tests, A/B timing).  The choice applies to forwards enqueued after the call: a captured CUDA graph keeps
 * replaying the kernel it was captured with. */
#define SPRL_EVALNET_PATH_AUTO 0
#define SPRL_EVALNET_PATH_STREAMING 1
#define SPRL_EVALNET_PATH_RESIDENT 2
int sprl_evalnet_set_path(sprl_evalnet* net, int path);
/* Arithmetic of the conv tower.  FP32_SPLIT (default; what every parity statement and the headline benchmark use): both
 * operands of every product are split into two fp16 terms, three MMAs per product, fp32 accumulation -- within 2e-6 of
 * the fp64 forward, the accuracy of the reference's fp32 LibTorch path.  FP16 (opt-in, resident kernel only): the hi
 * terms alone, one MMA per product, fp32 accumulation, fp32 bias / residual / head layers -- the "bf16/fp16 with fp32
 * accumulate" design point of an inference-only evaluator; about 1e-3 on logits.  It is NOT the reference's precision:
 * self-play statistics differ from an fp32 evaluator's, and a throughput measured with it is a different metric.
 * The mode applies to forwards enqueued after the call: a captured CUDA graph keeps the mode it was captured with. */
#define SPRL_EVALNET_PRECISION_FP32_SPLIT 0
#define SPRL_EVALNET_PRECISION_FP16 1
int sprl_evalnet_set_precision(sprl_evalnet* net, int precision);
/* Launches of the resident-weight kernel per forward (0: the streaming kernel is in use). */
int sprl_evalnet_phases(sprl_evalnet* net);
void sprl_evalnet_destroy(sprl_evalnet* net);

#ifdef __cplusplus
}
#endif
#endif
