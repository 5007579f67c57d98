// search.cuh -- device data model of the batched UCT search.
//
// One GPU warp owns one tree (one self-play game slot) and replays the
// reference's strictly sequential search semantics inside it
// (/root/reference/cpp/src/uct/UCTTree.hpp, uct/UCTNode.hpp); parallelism comes
// from thousands of independent trees.
//
// HBM layout.  Each tree owns two slabs (ping-pong for subtree compaction) of
// `cap_units` 16-byte units.  A node is a contiguous RECORD
//     [ header: HDR units ][ one 16-byte edge per legal action, ascending ]
// so that one pointer reaches the header and its edges in a single round trip.
// Unit 0 of a slab is the tree-level dummy edge that holds the root's own N/W
// (uct/UCTTree.hpp:301); the root record starts at unit 1.
//
//   header, 1-word games (Othello, Connect Four, Go 7x7), HDR = 3:
//     unit0 = { b0.lo, b0.hi, b1.lo, b1.hi }            stones of player ZERO / ONE
//     unit1 = { legal.lo, legal.hi, parent, own_edge }  unit indices within the slab
//     unit2 = { net_value, meta, aux, 0 }
//   header, 2-word games (Go 9x9), HDR = 5:
//     unit0 = b0, unit1 = b1, unit2 = legal, unit3 = { parent, own_edge, net_value, meta }, unit4 = { aux,0,0,0 }
//   edge  = { netP, W, N, (action << 24) | child }      child = 0: not created
//
// netP is the cached network prior (the reference's m_networkPolicy restricted to
// legal actions, uct/UCTNode.hpp:381); it survives re-rooting.  The reference's
// m_childPriors equals netP on every expanded node except the decision node with
// Dirichlet noise, whose mixed priors live in a per-tree array root_p[].
#pragma once
#include "games.cuh"
#include "rng.cuh"

namespace sprl {

enum { ST_IDLE = 0, ST_PLAYING = 1, ST_DONE = 2, ST_ERR_CAPACITY = 3, ST_ERR_MOVES = 4, ST_ERR_ACTION = 5 };

// meta word of a node header
#define META_NLEGAL(m) ((m) & 0xffu)
#define META_PLAYER(m) (((m) >> 8) & 1u)
#define META_TERMINAL(m) (((m) >> 9) & 1u)
#define META_WINNER(m) (((m) >> 10) & 3u)
#define META_EVALUATED (1u << 12)
#define META_EXPANDED (1u << 13)
#define META_PASS_LEGAL(m) (((m) >> 14) & 1u)
#define META_ACTION(m) (((m) >> 16) & 0xffu)

#define EDGE_CHILD(w) ((w) & 0x00ffffffu)
#define EDGE_ACTION(w) ((w) >> 24)

#define ROOT_UNIT 1u
#define SLAB_SLACK 64      // units kept free at the end of a slab (speculative loads)

struct TreeState {
    unsigned long long game_id;     // stream id of the game being played
    unsigned long long rng_ctr;     // next draw index of that stream
    u32 n_units;                    // bump pointer of the current slab
    u32 slab;                       // current slab (0/1)
    int traversals;                 // descents done for the current move
    int move_count;
    int status;                     // ST_*
    int n_queued;                   // leaves waiting for the evaluator
    long long game_index;           // index of the game inside the iteration
    u32 high_water;                 // max n_units seen
    u32 pad;
    // counters (summed on the host)
    unsigned long long sims, evals, moves, games;
    unsigned long long depth_sum, legal_sum, nodes_visited;
    unsigned long long leaves_terminal, leaves_gray, leaves_empty;
    unsigned long long leaves_duplicate;   // queued leaves that were already in the same batch's queue (quirk Q4): no evaluator row
};

struct AgentCfg {
    int evaluator, use_sym, init_q, pad;
    unsigned long long hash_salt;
};

// Values that change from one iteration / match to the next.  They live in device memory and are written on the
// engine's stream by sprl_begin_iteration / sprl_match_begin: kernel arguments are frozen into a captured CUDA graph,
// these are not, so one captured round serves every later iteration of the engine.
struct IterParams {
    long long num_games;
    unsigned long long first_game;
    unsigned long long game_stride;  // stream id of game i = first_game + i * game_stride
    u32 q_half;                      // first evaluator row of agent 1 (match play)
    // step-wise trees (sprl_begin_trees / sprl_search / sprl_advance): moves are made by the caller, a launch searches
    // a tree only while it has fewer than step_sims descents for the current move
    int stepwise;
    int step_sims;
    int step_single;                 // one searchAndGetLeaves batch per launch, whatever the evaluator (sprl_search_batch)
    AgentCfg agent[2];               // match play: the two sides
    // opening lines (sprl_set_openings; n_lines = 0: every game starts at the start position).  Stream id t plays line
    // t % n_lines (match play: (t / 2) % n_lines, so that both colour assignments play each line).  Line i has
    // open_off[i+1] - open_off[i] actions; its positions are open_rec[open_off[i] + i ..  open_off[i+1] + i]: the position
    // each of its actions is played in, then the position it ends in.  Read by init_game whenever a slot starts a game.
    long long n_lines;
    const long long* open_off;       // [n_lines + 1]
    const PosRec* open_rec;          // [open_off[n_lines] + n_lines]
};

struct EngineParams {
    // pools
    uint4* pool;                    // [n_slots][2][cap_units]
    unsigned long long cap_units;
    TreeState* trees;               // [n_slots]
    int n_slots;
    u32* q_leaf;                    // [n_slots][max_queue]
    unsigned char* q_sym;           // [n_slots][max_queue]
    u32* q_path;                    // [n_slots][max_queue][32] own edges of the nodes on the leaf's descent, root first
    unsigned char* q_plen;          // [n_slots][max_queue] how many of them (0: deeper than 32, back up by parent links)
    float* root_p;                  // [n_slots][ACTIONS] noised priors of the decision node, by edge slot
    // evaluator buffers (SPRL_EVAL_EXTERNAL).  Rows are handed out per launch, compactly: a tree with nq queued
    // leaves takes rows q_base[tree] .. +nq-1 (one atomicAdd on q_count), so the evaluator only computes the
    // q_rows[0] rows in use.  Match play: agent 1's rows start at q_half and are counted in q_count[1] / q_rows[1].
    float* nn_in;                   // [n_slots*max_queue][2H+1][R][C]
    const float* nn_logits;         // [n_slots*max_queue][A]
    const float* nn_value;          // [n_slots*max_queue]
    u32* q_count;                   // [2] rows handed out by the running launch
    u32* q_rows;                    // [2] rows of the previous launch: what the evaluator has to compute (set by k_flip)
    u32* q_base;                    // [n_slots] first row of a tree's queued leaves
    unsigned char* q_rowoff;        // [n_slots][max_queue] row of a queued leaf relative to q_base: a leaf queued twice in a batch
                                    //   (quirk Q4, uct/UCTTree.hpp:166-182: only its first evaluation is kept) gets ONE row
    u32 q_half;                     // first row of agent 1 (match play)            } host copies of the IterParams
    // per-game records, game-major: [num_games][max_moves]                            } fields: kernels read `iter`,
    long long num_games;             //                                                } never these
    unsigned long long first_game;
    unsigned long long game_stride;
    const IterParams* iter;          // device
    int max_moves;
    unsigned long long* rec_board;  // [..][2W]
    unsigned char* rec_player;      // [..]
    float* rec_pdf;                 // [..][A]
    int* rec_moves;                 // [num_games] searched moves (the opening's plies excluded) of a finished game, 0 before
    int* rec_open;                  // [num_games] plies of the game's opening line: its searched moves are recorded from there on
    unsigned char* rec_winner;      // [num_games]
    unsigned long long* rec_draws;  // [num_games]
    // optional per-move search statistics (parity tests)
    int record_stats;
    float* rec_N; float* rec_W; float* rec_P;   // [..][A]
    float* rec_root_N; float* rec_root_W;       // [..]
    int* rec_action; int* rec_trav;             // [..]
    // configuration (uct/UCTTree.hpp:38-42, selfplay/SelfPlay.hpp:52-56)
    int evaluator;
    unsigned long long seed;
    int sims, max_batch, max_queue;
    float dir_eps, dir_alpha, u_weight;
    int add_noise, use_sym, init_q;
    int fix_symmetry_mask;          // option (not the reference): mask the policy with the symmetrised legal mask
    int rounds_per_launch;
    unsigned long long* counters;   // [0] slots that finished all their games, [1] slots in error, [2] step-wise trees the running launch
                                    // still searched or that wait for evaluations, [3] the same of the previous launch (k_flip)
    // launch order of the trees (longest first): warp w of a launch serves tree order[parity][w].  Trees
    // that will finish a move in the next launch (sample + re-root = several times the work of a plain
    // search batch) are listed from the front, all others from the back, by the previous launch.
    u32* order;                     // [2][n_slots]
    u32* order_cnt;                 // [2][2] front / back fill counters of each list
    u32* order_parity;              // which list the next launch reads
    // re-rooting frontier (compact_into): per tree a FIFO of child links
    u32* cq;                        // [n_slots][cq_cap]
    u32 cq_cap;
};

// Match play (Evaluate.cpp:93-157): a game is served by a PAIR of trees, one per side; tree
// k * n_pairs + g belongs to agent k of pair g, so that the evaluator rows of one network are contiguous.
struct MatchParams {
    AgentCfg agent[2];               // host copy; kernels read IterParams::agent
    int n_pairs;
};

}  // namespace sprl
