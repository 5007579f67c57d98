// engine.cu -- host side of the self-play engine behind the C ABI of
// include/sprl_b200.h: owns the device pools, enqueues the search kernels of
// search.cu on one CUDA stream, turns the per-game records into the reference's
// sample arrays and writes them as .npy.
#include <algorithm>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "search.cuh"

namespace sprl {
void search_launch_begin(int game, const EngineParams& p, cudaStream_t s);
void search_launch_round(int game, const EngineParams& p, cudaStream_t s);
void search_launch_emit(int game, const EngineParams& p, long long g0, long long n_games, const long long* row0, int S, float* st, float* di,
                        float* ou, cudaStream_t s);
void search_launch_match_begin(int game, const EngineParams& p, const MatchParams& m, cudaStream_t s);
void search_launch_match_round(int game, const EngineParams& p, const MatchParams& m, cudaStream_t s);
void search_launch_tree_stats(int game, const EngineParams& p, int n, float* N, float* W, float* P, float* rn, float* rw, signed char* pl,
                              signed char* te, signed char* wi, int* tr, signed char* mk, int* qu, cudaStream_t s);
void search_launch_tree_advance(int game, const EngineParams& p, int n, const int* actions, cudaStream_t s);
int search_header_units(int game);
void env_launch_lines(int game, int n_lines, const long long* off, const int* actions, PosRec* rec, u64* hist, int* bad,
                      cudaStream_t s);
}  // namespace sprl

using namespace sprl;

struct sprl_engine {
    sprl_config cfg;
    sprl_game_info gi;
    EngineParams p;
    cudaStream_t stream = nullptr;
    int words = 1;                  // 64-bit words per colour
    int64_t num_games = 0;          // of the running / last iteration
    int64_t active_slots = 0;
    bool iteration_open = false;
    bool match_open = false;        // the open iteration is a match (pairs of trees)
    MatchParams match;
    IterParams* d_iter = nullptr;   // device copy of the per-iteration values (search.cuh)
    bool stepwise = false;          // the open iteration is a set of step-wise trees (sprl_begin_trees)
    int step_sims = 0;
    bool step_single = false;
    // opening lines of the games the next begin starts (sprl_set_openings; IterParams describes the layout)
    int64_t n_lines = 0;
    long long* d_open_off = nullptr;
    PosRec* d_open_rec = nullptr;
    unsigned char* d_tree_io = nullptr;     // staging of sprl_root_stats / sprl_advance, sized for num_slots trees
    // Streamed sample output (sprl_stream_samples): finished games are embedded and copied to the caller's (pinned) host
    // arrays while the others still play.  Two copy streams, each with its own staging buffers of `rows` sample rows.
    struct StreamOut {
        bool active = false, registered = false;
        float *h_states = nullptr, *h_dists = nullptr, *h_outcomes = nullptr;
        int64_t cap = 0;                    // sample rows the host arrays hold
        int64_t games_done = 0, rows_done = 0;
        int64_t rows = 0;                   // staging capacity
        cudaStream_t stream[2] = { nullptr, nullptr };
        float* d_states[2] = { nullptr, nullptr }; float* d_dists[2] = { nullptr, nullptr }; float* d_outcomes[2] = { nullptr, nullptr };
        long long* d_row0 = nullptr;        // [max_games]
        int which = 0;
        bool overflow = false;
        uint64_t chunks = 0;                // chunks copied while games were still playing (reported by sprl_stream_info)
    } so;
    bool failed = false;            // sticky CUDA error
    uint64_t launches = 0;
    uint64_t device_bytes = 0;
    std::vector<void*> allocations;
    // sample output (device), sized on demand
    float* d_states = nullptr; float* d_dists = nullptr; float* d_outcomes = nullptr;
    long long* d_row0 = nullptr;
    int64_t sample_cap = 0;
    // counters snapshot at reset
    sprl_stats base;
    std::vector<int> h_moves;

    // Every pool sits between two 256-byte guard bands filled with a pattern (sprl_debug_check_guards): the kernels index
    // their pools with tree-, queue- and game-relative offsets, and compute-sanitizer is not available on every box.
    static constexpr size_t GUARD = 256;
    struct Pool { unsigned char* base; size_t bytes; };
    std::vector<Pool> pools;
    template <typename T> int alloc(T** out, size_t count, bool zero) {
        void* ptr = nullptr;
        size_t bytes = (std::max<size_t>(count, 1) * sizeof(T) + 255) / 256 * 256;
        cudaError_t err = cudaMalloc(&ptr, bytes + 2 * GUARD);
        if (err != cudaSuccess) return fail(SPRL_E_CAPACITY, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(err));
        unsigned char* base = (unsigned char*)ptr;
        err = cudaMemset(base, 0xA5, GUARD);
        if (err == cudaSuccess) err = cudaMemset(base + GUARD + bytes, 0xA5, GUARD);
        if (err == cudaSuccess && zero) err = cudaMemset(base + GUARD, 0, bytes);
        if (err != cudaSuccess) return fail(SPRL_E_CUDA, "cudaMemset: %s", cudaGetErrorString(err));
        allocations.push_back(ptr);
        pools.push_back(Pool{ base, bytes });
        device_bytes += bytes + 2 * GUARD;
        *out = (T*)(base + GUARD);
        return SPRL_OK;
    }
    // frees one pool taken by alloc()
    void release(void* ptr) {
        if (!ptr) return;
        unsigned char* base = (unsigned char*)ptr - GUARD;
        for (size_t i = 0; i < pools.size(); ++i)
            if (pools[i].base == base) { device_bytes -= pools[i].bytes + 2 * GUARD; pools.erase(pools.begin() + i); break; }
        allocations.erase(std::remove(allocations.begin(), allocations.end(), (void*)base), allocations.end());
        cudaFree(base);
    }
    void free_all() {
        for (void* q : allocations) cudaFree(q);
        allocations.clear();
        if (d_states) cudaFree(d_states);
        if (d_dists) cudaFree(d_dists);
        if (d_outcomes) cudaFree(d_outcomes);
        if (d_row0) cudaFree(d_row0);
        d_states = d_dists = d_outcomes = nullptr; d_row0 = nullptr;
        stream_out_release();
    }
    void stream_out_unregister() {
        if (so.registered) { cudaHostUnregister(so.h_states); cudaHostUnregister(so.h_dists); cudaHostUnregister(so.h_outcomes); }
        so.registered = false;
    }
    void stream_out_release() {
        stream_out_unregister();
        for (int k = 0; k < 2; ++k) {
            if (so.stream[k]) cudaStreamDestroy(so.stream[k]);
            if (so.d_states[k]) cudaFree(so.d_states[k]);
            if (so.d_dists[k]) cudaFree(so.d_dists[k]);
            if (so.d_outcomes[k]) cudaFree(so.d_outcomes[k]);
        }
        if (so.d_row0) cudaFree(so.d_row0);
        so = StreamOut();
    }
};

#define ENGINE_CHECK(e)                                                                   \
    do {                                                                                  \
        if (!(e)) return fail(SPRL_E_INVALID, "null engine");                             \
        if ((e)->failed) return fail(SPRL_E_CUDA, "engine is in a failed state: %s", last_error_ref().c_str()); \
        cudaError_t se__ = cudaSetDevice((e)->cfg.device);                                \
        if (se__ != cudaSuccess) return fail(SPRL_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(se__)); \
    } while (0)

#define ENGINE_CUDA(e, expr)                                                              \
    do {                                                                                  \
        cudaError_t err__ = (expr);                                                       \
        if (err__ != cudaSuccess) {                                                       \
            (e)->failed = true;                                                           \
            return fail(SPRL_E_CUDA, "%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(err__)); \
        }                                                                                 \
    } while (0)

static int sum_tree_stats(sprl_engine* e, sprl_stats* out) {
    std::vector<TreeState> ts(e->cfg.num_slots);
    ENGINE_CUDA(e, cudaMemcpyAsync(ts.data(), e->p.trees, ts.size() * sizeof(TreeState), cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    memset(out, 0, sizeof(*out));
    for (const TreeState& t : ts) {
        out->sims += t.sims; out->evals += t.evals; out->moves += t.moves; out->games += t.games;
        out->depth_sum += t.depth_sum; out->legal_sum += t.legal_sum; out->nodes_visited += t.nodes_visited;
        out->leaves_terminal += t.leaves_terminal; out->leaves_gray += t.leaves_gray; out->leaves_empty += t.leaves_empty;
        out->leaves_duplicate += t.leaves_duplicate;
        out->units_high_water = std::max<uint64_t>(out->units_high_water, t.high_water);
    }
    out->units_per_tree = e->p.cap_units;
    out->launches = e->launches;
    out->device_bytes = e->device_bytes;
    return SPRL_OK;
}

// Publishes the per-iteration values on the stream (see IterParams: a captured graph must not freeze them).
static int push_iter_params(sprl_engine* e) {
    IterParams it;
    memset(&it, 0, sizeof(it));
    it.num_games = e->p.num_games; it.first_game = e->p.first_game; it.game_stride = e->p.game_stride; it.q_half = e->p.q_half;
    it.stepwise = e->stepwise ? 1 : 0; it.step_sims = e->step_sims; it.step_single = e->step_single ? 1 : 0;
    it.agent[0] = e->match.agent[0]; it.agent[1] = e->match.agent[1];
    it.n_lines = e->n_lines; it.open_off = e->d_open_off; it.open_rec = e->d_open_rec;
    cudaError_t err = cudaMemcpyAsync(e->d_iter, &it, sizeof(it), cudaMemcpyHostToDevice, e->stream);   // pageable source: staged before the call returns
    if (err != cudaSuccess) { e->failed = true; return fail(SPRL_E_CUDA, "cudaMemcpyAsync of the iteration parameters failed: %s", cudaGetErrorString(err)); }
    return SPRL_OK;
}

static int check_tree_options(int game, int evaluator, int init_q) {
    if (evaluator < SPRL_EVAL_UNIFORM || evaluator > SPRL_EVAL_OTHELLO_HEURISTIC) return fail(SPRL_E_INVALID, "unknown evaluator %d", evaluator);
    if (evaluator == SPRL_EVAL_OTHELLO_HEURISTIC && game != SPRL_GAME_OTHELLO)
        return fail(SPRL_E_INVALID, "SPRL_EVAL_OTHELLO_HEURISTIC evaluates Othello positions only");
    if (init_q < SPRL_INITQ_ZERO || init_q > SPRL_INITQ_DROP_PARENT) return fail(SPRL_E_INVALID, "unknown init_q %d", init_q);
    return SPRL_OK;
}

extern "C" {

int sprl_default_config(int game, sprl_config* cfg) {
    if (!cfg) return fail(SPRL_E_INVALID, "null config");
    sprl_game_info gi;
    int rc = sprl_game_info_get(game, &gi);
    if (rc) return rc;
    memset(cfg, 0, sizeof(*cfg));
    cfg->device = 0; cfg->game = game; cfg->evaluator = SPRL_EVAL_UNIFORM; cfg->seed = 0;
    cfg->num_slots = 1024;
    cfg->dir_eps = 0.25f; cfg->u_weight = 1.1f;           // constants.hpp:6
    cfg->add_noise = 1; cfg->use_sym = 1; cfg->init_q = SPRL_INITQ_PARENT;
    switch (game) {
    case SPRL_GAME_OTHELLO: cfg->sims = 8192; cfg->max_batch = 8; cfg->max_queue = 4; cfg->dir_alpha = 0.3f; break;   // OTHWorker.cpp:23-28
    case SPRL_GAME_C4: cfg->sims = 512; cfg->max_batch = 8; cfg->max_queue = 4; cfg->dir_alpha = 0.5f; break;        // C4Worker.cpp:22-27
    default: cfg->sims = 32768; cfg->max_batch = 16; cfg->max_queue = 8; cfg->dir_alpha = 0.2f; break;               // GoWorker.cpp:22-27
    }
    cfg->units_per_tree = 0; cfg->max_games = 0; cfg->record_stats = 0; cfg->rounds_per_launch = 0;
    return SPRL_OK;
}

int sprl_create(const sprl_config* cfg, sprl_engine** out) {
    if (!cfg || !out) return fail(SPRL_E_INVALID, "null argument");
    *out = nullptr;
    sprl_game_info gi;
    int rc = sprl_game_info_get(cfg->game, &gi);
    if (rc) return rc;
    if (cfg->num_slots <= 0 || cfg->sims <= 0 || cfg->max_batch <= 0 || cfg->max_queue <= 0)
        return fail(SPRL_E_INVALID, "num_slots, sims, max_batch and max_queue must be positive");
    if (cfg->max_queue > 255) return fail(SPRL_E_INVALID, "max_queue is limited to 255 leaves per tree and batch");
    rc = check_tree_options(cfg->game, cfg->evaluator, cfg->init_q);
    if (rc) return rc;
    if (!(cfg->dir_alpha > 0.0f) && cfg->add_noise) return fail(SPRL_E_INVALID, "dir_alpha must be positive");
    rc = use_device(cfg->device);
    if (rc) return rc;

    sprl_engine* e = new sprl_engine();
    e->cfg = *cfg;
    e->gi = gi;
    e->words = gi.cells <= 64 ? 1 : 2;
    memset(&e->base, 0, sizeof(e->base));
    if (e->cfg.max_games <= 0) e->cfg.max_games = e->cfg.num_slots;
    if (e->cfg.rounds_per_launch <= 0) e->cfg.rounds_per_launch = 8;
    const int hdr = search_header_units(cfg->game);
    if (e->cfg.units_per_tree <= 0) {
        // A search adds at most one node per descent and re-rooting keeps only the chosen subtree, so
        // the live tree is bounded by sims / (1 - kept fraction); 6x covers kept fractions up to ~0.83
        // (Connect Four with a uniform evaluator keeps the most).  A record = header + one edge per
        // legal action; `typical` is a generous per-game average of the latter.
        int typical = cfg->game == SPRL_GAME_OTHELLO ? 12 : (cfg->game == SPRL_GAME_C4 ? 7 : (cfg->game == SPRL_GAME_GO7 ? 45 : 75));
        int64_t nodes = 6 * (int64_t)(cfg->sims + cfg->max_batch) + 64;
        e->cfg.units_per_tree = std::max<int64_t>(4096, nodes * (hdr + typical));
    }
    if (cfg->units_per_tree > (1 << 24) - 1) {                                               // child index is 24 bits
        delete e;
        return fail(SPRL_E_INVALID, "units_per_tree = %lld exceeds the 24-bit child index (at most %d units of 16 bytes per slab)", (long long)cfg->units_per_tree, (1 << 24) - 1);
    }
    if (e->cfg.units_per_tree > (1 << 24) - 1) {
        // derived from the search budget (the reference's Go worker asks for 32,768 descents per move): the slab stops
        // at the index width, and a tree that outgrows it reports SPRL_E_CAPACITY when it happens
        fprintf(stderr, "sprl_create: sims = %d asks for %lld units per tree, clamped to %d (24-bit child index, %.2f GB per tree)\n",
                cfg->sims, (long long)e->cfg.units_per_tree, (1 << 24) - 1, 2.0 * 16.0 * ((1 << 24) - 1) / 1e9);
        e->cfg.units_per_tree = (1 << 24) - 1;
    }
    if (e->cfg.units_per_tree < 2 * (hdr + gi.actions) + SLAB_SLACK + 2) { delete e; return fail(SPRL_E_INVALID, "units_per_tree too small"); }

    EngineParams& p = e->p;
    memset(&p, 0, sizeof(p));
    p.cap_units = (unsigned long long)e->cfg.units_per_tree;
    p.n_slots = cfg->num_slots;
    p.max_moves = gi.max_plies;
    p.evaluator = cfg->evaluator; p.seed = cfg->seed;
    p.sims = cfg->sims; p.max_batch = cfg->max_batch; p.max_queue = cfg->max_queue;
    p.dir_eps = cfg->dir_eps; p.dir_alpha = cfg->dir_alpha; p.u_weight = cfg->u_weight;
    p.add_noise = cfg->add_noise; p.use_sym = cfg->use_sym; p.init_q = cfg->init_q;
    p.fix_symmetry_mask = cfg->fix_symmetry_mask ? 1 : 0;
    p.rounds_per_launch = (cfg->evaluator == SPRL_EVAL_EXTERNAL) ? 1 : e->cfg.rounds_per_launch;
    p.record_stats = cfg->record_stats;
    p.game_stride = 1;

    const size_t S = (size_t)cfg->num_slots, MG = (size_t)e->cfg.max_games, MM = (size_t)gi.max_plies, A = (size_t)gi.actions;
    rc = e->alloc(&p.pool, S * 2 * p.cap_units, false);
    if (rc) {
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const double per_tree = 2.0 * 16.0 * (double)p.cap_units;
        rc = fail(SPRL_E_CAPACITY, "the tree slabs do not fit: %d slots x %.1f MB per tree (2 slabs of %llu units) = %.1f GB, %.1f GB free on the device; "
                  "lower num_slots (about %lld fit) or units_per_tree", cfg->num_slots, per_tree / 1e6, p.cap_units, per_tree * S / 1e9, free_b / 1e9,
                  (long long)(0.9 * free_b / per_tree));
    }
    if (!rc) rc = e->alloc(&p.trees, S, true);
    if (!rc) rc = e->alloc(&p.q_leaf, S * cfg->max_queue, true);
    if (!rc) rc = e->alloc(&p.q_sym, S * cfg->max_queue, true);
    if (!rc) rc = e->alloc(&p.q_path, S * cfg->max_queue * 32, false);
    if (!rc) rc = e->alloc(&p.q_plen, S * cfg->max_queue, true);
    if (!rc) rc = e->alloc(&p.q_count, 2, true);
    if (!rc) rc = e->alloc(&p.q_rows, 2, true);
    if (!rc) rc = e->alloc(&p.q_base, S, true);
    if (!rc) rc = e->alloc(&p.q_rowoff, S * cfg->max_queue, true);
    if (!rc) rc = e->alloc(&p.root_p, S * A, true);
    if (!rc) rc = e->alloc(&p.rec_board, MG * MM * 2 * e->words, true);
    if (!rc) rc = e->alloc(&p.rec_player, MG * MM, true);
    if (!rc) rc = e->alloc(&p.rec_pdf, MG * MM * A, false);
    if (!rc) rc = e->alloc(&p.rec_moves, MG, true);
    if (!rc) rc = e->alloc(&p.rec_open, MG, true);
    if (!rc) rc = e->alloc(&p.rec_winner, MG, true);
    if (!rc) rc = e->alloc(&p.rec_draws, MG, true);
    if (!rc) rc = e->alloc(&p.counters, 4, true);
    p.cq_cap = (u32)(p.cap_units / (unsigned long long)hdr + 1);
    if (!rc) rc = e->alloc(&p.cq, S * p.cq_cap, false);
    if (!rc) rc = e->alloc(&p.order, S * 2, true);
    if (!rc) rc = e->alloc(&p.order_cnt, 4, true);
    if (!rc) rc = e->alloc(&p.order_parity, 1, true);
    if (!rc) rc = e->alloc(&e->d_iter, 1, true);
    p.iter = e->d_iter;
    memset(&e->match, 0, sizeof(e->match));
    if (!rc && cfg->record_stats) {
        rc = e->alloc(&p.rec_N, MG * MM * A, false);
        if (!rc) rc = e->alloc(&p.rec_W, MG * MM * A, false);
        if (!rc) rc = e->alloc(&p.rec_P, MG * MM * A, false);
        if (!rc) rc = e->alloc(&p.rec_root_N, MG * MM, false);
        if (!rc) rc = e->alloc(&p.rec_root_W, MG * MM, false);
        if (!rc) rc = e->alloc(&p.rec_action, MG * MM, false);
        if (!rc) rc = e->alloc(&p.rec_trav, MG * MM, false);
    }
    if (rc) { e->free_all(); delete e; return rc; }
    *out = e;
    return SPRL_OK;
}

void sprl_destroy(sprl_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaDeviceSynchronize();
    e->free_all();
    delete e;
}

int sprl_set_stream(sprl_engine* e, void* cuda_stream) {
    ENGINE_CHECK(e);
    e->stream = (cudaStream_t)cuda_stream;
    return SPRL_OK;
}

int sprl_bind_eval_buffers(sprl_engine* e, float* d_in, const float* d_logits, const float* d_value) {
    ENGINE_CHECK(e);
    if (e->cfg.evaluator != SPRL_EVAL_EXTERNAL) return fail(SPRL_E_STATE, "engine was not created with SPRL_EVAL_EXTERNAL");
    if (!d_in || !d_logits || !d_value) return fail(SPRL_E_INVALID, "null evaluator buffer");
    e->p.nn_in = d_in; e->p.nn_logits = d_logits; e->p.nn_value = d_value;
    return SPRL_OK;
}

int sprl_set_game_stride(sprl_engine* e, uint64_t stride) {
    ENGINE_CHECK(e);
    if (stride == 0) return fail(SPRL_E_INVALID, "stride must be positive");
    e->p.game_stride = stride;
    return SPRL_OK;
}

int sprl_eval_rows(sprl_engine* e, const uint32_t** d_rows) {
    ENGINE_CHECK(e);
    if (!d_rows) return fail(SPRL_E_INVALID, "null output");
    *d_rows = e->p.q_rows;
    return SPRL_OK;
}

int64_t sprl_eval_batch(const sprl_engine* e) { return e ? (int64_t)e->cfg.num_slots * e->cfg.max_queue : 0; }

int sprl_set_openings(sprl_engine* e, int64_t n_lines, const int64_t* h_offsets, const int32_t* h_actions) {
    NvtxRange nvtx_range("sprl_set_openings");
    ENGINE_CHECK(e);
    if (n_lines < 0 || n_lines > (1 << 30)) return fail(SPRL_E_INVALID, "n_lines = %lld is out of range", (long long)n_lines);
    if (n_lines > 0 && !h_offsets) return fail(SPRL_E_INVALID, "null offsets");
    if (e->iteration_open) {
        // slots start games from the table until the last game has started: it changes only when no game is playing
        unsigned long long c[4] = { 0, 0, 0, 0 };
        ENGINE_CUDA(e, cudaMemcpyAsync(c, e->p.counters, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
        ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
        if (e->active_slots - (int64_t)c[0] - (int64_t)c[1] > 0)
            return fail(SPRL_E_STATE, "openings cannot change while an iteration, a match or a set of step-wise trees is still playing");
    }
    int64_t total = 0;
    if (n_lines > 0) {
        if (h_offsets[0] != 0) return fail(SPRL_E_INVALID, "h_offsets[0] must be 0");
        for (int64_t i = 0; i < n_lines; ++i)
            if (h_offsets[i + 1] < h_offsets[i]) return fail(SPRL_E_INVALID, "h_offsets must not decrease (line %lld)", (long long)i);
        total = h_offsets[n_lines];
        if (total > (1 << 30)) return fail(SPRL_E_INVALID, "the lines hold %lld actions, more than %d", (long long)total, 1 << 30);
        if (total > 0 && !h_actions) return fail(SPRL_E_INVALID, "null actions");
    }
    // every line is replayed once, on the device; the old table stays in use until the new one has been checked
    long long* d_off = nullptr;
    PosRec* d_rec = nullptr;
    if (n_lines > 0) {
        int rc = e->alloc(&d_off, (size_t)n_lines + 1, false);
        if (!rc) rc = e->alloc(&d_rec, (size_t)(total + n_lines), false);
        if (rc) { e->release(d_off); return rc; }
        DeviceBuf<int> d_act, d_bad;
        DeviceBuf<u64> d_hist;
        cudaError_t err = d_act.alloc((size_t)std::max<int64_t>(total, 1));
        if (err == cudaSuccess) err = d_bad.alloc((size_t)n_lines);
        if (err == cudaSuccess) err = d_hist.alloc((size_t)std::max<int64_t>(total, 1) * 2 * e->words);
        if (err == cudaSuccess) err = cudaMemcpyAsync(d_off, h_offsets, ((size_t)n_lines + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess && total > 0) err = cudaMemcpyAsync(d_act.p, h_actions, (size_t)total * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) {
            env_launch_lines(e->cfg.game, (int)n_lines, d_off, d_act.p, d_rec, d_hist.p, d_bad.p, e->stream);
            e->launches += 1;
            err = cudaGetLastError();
        }
        std::vector<int> bad((size_t)n_lines);
        std::vector<PosRec> rec((size_t)(total + n_lines));
        if (err == cudaSuccess) err = cudaMemcpyAsync(bad.data(), d_bad.p, bad.size() * sizeof(int), cudaMemcpyDeviceToHost, e->stream);
        if (err == cudaSuccess) err = cudaMemcpyAsync(rec.data(), d_rec, rec.size() * sizeof(PosRec), cudaMemcpyDeviceToHost, e->stream);
        if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
        if (err != cudaSuccess) {
            e->failed = true;
            return fail(SPRL_E_CUDA, "replay of the opening lines failed: %s", cudaGetErrorString(err));
        }
        for (int64_t i = 0; i < n_lines; ++i) {
            const int64_t ply = bad[i] >= 0 ? bad[i] : h_offsets[i + 1] - h_offsets[i];     // where the replay stopped
            int rc = SPRL_OK;
            if (rec[(size_t)(h_offsets[i] + i + ply)].terminal)
                rc = fail(SPRL_E_INVALID, "opening line %lld reaches a terminal position at ply %lld: a game must have a move left to search",
                          (long long)i, (long long)ply);
            else if (bad[i] >= 0)
                rc = fail(SPRL_E_INVALID, "opening line %lld: action %d at ply %lld is not legal in the position it is played in",
                          (long long)i, h_actions[h_offsets[i] + ply], (long long)ply);
            if (rc) { e->release(d_rec); e->release(d_off); return rc; }
        }
    }
    e->release(e->d_open_rec);
    e->release(e->d_open_off);
    e->d_open_off = d_off;
    e->d_open_rec = d_rec;
    e->n_lines = n_lines;
    return SPRL_OK;
}

int sprl_begin_iteration(sprl_engine* e, uint64_t first_game, int64_t num_games) {
    NvtxRange nvtx_range("sprl_begin_iteration");
    ENGINE_CHECK(e);
    if (num_games <= 0) return fail(SPRL_E_INVALID, "num_games must be positive");
    if (num_games > e->cfg.max_games) return fail(SPRL_E_CAPACITY, "num_games %lld exceeds max_games %lld", (long long)num_games, (long long)e->cfg.max_games);
    e->p.first_game = first_game;
    e->p.num_games = num_games;
    e->num_games = num_games;
    e->active_slots = std::min<int64_t>(num_games, e->cfg.num_slots);
    e->p.q_half = 0;
    e->stepwise = false;
    e->so.games_done = e->so.rows_done = 0; e->so.overflow = false; e->so.which = 0;
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.q_count, 0, 2 * sizeof(u32), e->stream));
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.q_rows, 0, 2 * sizeof(u32), e->stream));
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.counters, 0, 4 * sizeof(unsigned long long), e->stream));
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_moves, 0, (size_t)e->cfg.max_games * sizeof(int), e->stream));
    if (e->cfg.record_stats) {
        // only legal actions are written per move; the rest of each [A] row must read as 0
        const size_t bytes = (size_t)e->cfg.max_games * e->p.max_moves * e->gi.actions * sizeof(float);
        ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_N, 0, bytes, e->stream));
        ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_W, 0, bytes, e->stream));
        ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_P, 0, bytes, e->stream));
    }
    { int rc = push_iter_params(e); if (rc) return rc; }
    search_launch_begin(e->cfg.game, e->p, e->stream);
    e->launches += 1;
    ENGINE_CUDA(e, cudaGetLastError());
    e->iteration_open = true;
    e->match_open = false;
    return SPRL_OK;
}

static int load_game_moves(sprl_engine* e, int64_t* n_moves);

int sprl_match_begin(sprl_engine* e, const sprl_agent_config* h_agents, uint64_t first_game, int64_t num_games) {
    NvtxRange nvtx_range("sprl_match_begin");
    ENGINE_CHECK(e);
    if (!h_agents) return fail(SPRL_E_INVALID, "null agents");
    if (num_games <= 0) return fail(SPRL_E_INVALID, "num_games must be positive");
    if (num_games > e->cfg.max_games) return fail(SPRL_E_CAPACITY, "num_games %lld exceeds max_games %lld", (long long)num_games, (long long)e->cfg.max_games);
    if (e->cfg.num_slots < 2) return fail(SPRL_E_INVALID, "a match needs two tree slots per game");
    bool external = false;
    for (int k = 0; k < 2; ++k) {
        int rc = check_tree_options(e->cfg.game, h_agents[k].evaluator, h_agents[k].init_q);
        if (rc) return rc;
        external = external || h_agents[k].evaluator == SPRL_EVAL_EXTERNAL;
        e->match.agent[k].evaluator = h_agents[k].evaluator;
        e->match.agent[k].use_sym = h_agents[k].use_sym;
        e->match.agent[k].init_q = h_agents[k].init_q;
        e->match.agent[k].pad = k;                       // which half of the evaluator batch
        e->match.agent[k].hash_salt = h_agents[k].hash_salt;
    }
    if (external && e->cfg.evaluator != SPRL_EVAL_EXTERNAL)
        return fail(SPRL_E_STATE, "an agent with SPRL_EVAL_EXTERNAL needs an engine created with SPRL_EVAL_EXTERNAL");
    if (external && !e->p.nn_in) return fail(SPRL_E_STATE, "evaluator buffers are not bound");
    e->match.n_pairs = e->cfg.num_slots / 2;
    e->stepwise = false;
    e->p.first_game = first_game;
    e->p.num_games = num_games;
    e->num_games = num_games;
    e->active_slots = std::min<int64_t>(num_games, e->match.n_pairs);
    e->p.q_half = (u32)e->match.n_pairs * (u32)e->cfg.max_queue;
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.q_count, 0, 2 * sizeof(u32), e->stream));
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.q_rows, 0, 2 * sizeof(u32), e->stream));
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.counters, 0, 4 * sizeof(unsigned long long), e->stream));
    ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_moves, 0, (size_t)e->cfg.max_games * sizeof(int), e->stream));
    if (e->cfg.record_stats) {
        const size_t bytes = (size_t)e->cfg.max_games * e->p.max_moves * e->gi.actions * sizeof(float);
        ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_N, 0, bytes, e->stream));
        ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_W, 0, bytes, e->stream));
        ENGINE_CUDA(e, cudaMemsetAsync(e->p.rec_P, 0, bytes, e->stream));
    }
    { int rc = push_iter_params(e); if (rc) return rc; }
    search_launch_match_begin(e->cfg.game, e->p, e->match, e->stream);
    e->launches += 1;
    ENGINE_CUDA(e, cudaGetLastError());
    e->iteration_open = true;
    e->match_open = true;
    return SPRL_OK;
}

int sprl_match_results(sprl_engine* e, int64_t cap_games, int8_t* h_winner, int32_t* h_moves, uint64_t* h_draws,
                       int64_t* wins, int64_t* draws) {
    ENGINE_CHECK(e);
    if (!e->iteration_open || !e->match_open) return fail(SPRL_E_STATE, "no match has been run");
    if (cap_games < e->num_games && (h_winner || h_moves || h_draws))
        return fail(SPRL_E_CAPACITY, "%lld games do not fit the caller's capacity %lld", (long long)e->num_games, (long long)cap_games);
    int64_t total = 0;
    int rc = load_game_moves(e, &total);
    if (rc) return rc;
    std::vector<unsigned char> w((size_t)e->num_games);
    ENGINE_CUDA(e, cudaMemcpyAsync(w.data(), e->p.rec_winner, w.size(), cudaMemcpyDeviceToHost, e->stream));
    if (h_draws) ENGINE_CUDA(e, cudaMemcpyAsync(h_draws, e->p.rec_draws, (size_t)e->num_games * 8, cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    int64_t tally[2] = { 0, 0 }, none = 0;
    for (int64_t g = 0; g < e->num_games; ++g) {
        const int winner = (int)w[g] - 1;                       // device encoding: 0 none, 1 ZERO, 2 ONE
        if (h_winner) h_winner[g] = (int8_t)winner;
        if (h_moves) h_moves[g] = e->h_moves[g];
        if (e->h_moves[g] == 0) continue;                        // not played
        const uint64_t id = e->p.first_game + (uint64_t)g * e->p.game_stride;
        if (winner < 0) none += 1;
        else tally[(id & 1ULL) ? 1 - winner : winner] += 1;     // Evaluate.cpp:139-153
    }
    if (wins) { wins[0] = tally[0]; wins[1] = tally[1]; }
    if (draws) *draws = none;
    return SPRL_OK;
}

// Streamed output: embeds the samples of the games that have finished since the last call -- the contiguous prefix of the
// iteration's games, because a game's rows follow those of all earlier games -- and copies them to the host arrays, on the
// copy streams.  The caller has synchronised the engine's stream (the records of finished games are final).
static int stream_out_advance(sprl_engine* e) {
    sprl_engine::StreamOut& so = e->so;
    if (so.overflow) return SPRL_OK;
    int64_t total = 0;
    int rc = load_game_moves(e, &total);                // rec_moves[g] > 0 <=> game g is over
    if (rc) return rc;
    const int S = e->cfg.use_sym ? e->gi.nsym : 1;
    const size_t row = (size_t)(2 * e->gi.history + 1) * e->gi.cells, A = (size_t)e->gi.actions;
    int64_t g = so.games_done;
    while (g < e->num_games) {
        // the next chunk: finished games from g on, as many as the staging buffers hold
        int64_t g1 = g, rows = 0;
        std::vector<long long> row0;
        while (g1 < e->num_games && e->h_moves[g1] > 0 && rows + (int64_t)e->h_moves[g1] * S <= so.rows) {
            row0.push_back(rows);
            rows += (int64_t)e->h_moves[g1] * S;
            ++g1;
        }
        if (g1 == g) {
            if (g < e->num_games && e->h_moves[g] > 0) return fail(SPRL_E_CAPACITY, "a single game's samples exceed the staging buffer");
            break;                                      // game g is still being played
        }
        if (so.rows_done + rows > so.cap) { so.overflow = true; break; }     // reported by sprl_collect_samples
        const int w = so.which;
        so.which ^= 1;
        cudaStream_t cs = so.stream[w];
        ENGINE_CUDA(e, cudaMemcpyAsync(so.d_row0 + g, row0.data(), row0.size() * sizeof(long long), cudaMemcpyHostToDevice, cs));   // pageable: staged at once
        search_launch_emit(e->cfg.game, e->p, g, g1 - g, so.d_row0, S, so.d_states[w], so.d_dists[w], so.d_outcomes[w], cs);
        e->launches += 1;
        ENGINE_CUDA(e, cudaGetLastError());
        ENGINE_CUDA(e, cudaMemcpyAsync(so.h_states + (size_t)so.rows_done * row, so.d_states[w], (size_t)rows * row * sizeof(float), cudaMemcpyDeviceToHost, cs));
        ENGINE_CUDA(e, cudaMemcpyAsync(so.h_dists + (size_t)so.rows_done * A, so.d_dists[w], (size_t)rows * A * sizeof(float), cudaMemcpyDeviceToHost, cs));
        ENGINE_CUDA(e, cudaMemcpyAsync(so.h_outcomes + (size_t)so.rows_done, so.d_outcomes[w], (size_t)rows * sizeof(float), cudaMemcpyDeviceToHost, cs));
        so.rows_done += rows;
        g = g1;
    }
    so.games_done = g;
    return SPRL_OK;
}

int sprl_stream_samples(sprl_engine* e, int64_t cap_samples, float* h_states, float* h_distributions, float* h_outcomes, int pin) {
    ENGINE_CHECK(e);
    sprl_engine::StreamOut& so = e->so;
    if (e->iteration_open && so.active && so.games_done > 0) ENGINE_CUDA(e, cudaDeviceSynchronize());
    e->stream_out_unregister();
    so.active = false;
    if (!h_states && !h_distributions && !h_outcomes) return SPRL_OK;          // streaming off
    if (!h_states || !h_distributions || !h_outcomes || cap_samples <= 0) return fail(SPRL_E_INVALID, "sprl_stream_samples needs the three host arrays and their capacity");
    const int S = e->cfg.use_sym ? e->gi.nsym : 1;
    const size_t row = (size_t)(2 * e->gi.history + 1) * e->gi.cells, A = (size_t)e->gi.actions;
    if (!so.stream[0]) {
        so.rows = std::max<int64_t>(1 << 16, (int64_t)e->p.max_moves * S);      // >= one game of maximal length
        for (int k = 0; k < 2; ++k) {
            ENGINE_CUDA(e, cudaStreamCreateWithFlags(&so.stream[k], cudaStreamNonBlocking));
            ENGINE_CUDA(e, cudaMalloc((void**)&so.d_states[k], (size_t)so.rows * row * sizeof(float)));
            ENGINE_CUDA(e, cudaMalloc((void**)&so.d_dists[k], (size_t)so.rows * A * sizeof(float)));
            ENGINE_CUDA(e, cudaMalloc((void**)&so.d_outcomes[k], (size_t)so.rows * sizeof(float)));
        }
        ENGINE_CUDA(e, cudaMalloc((void**)&so.d_row0, (size_t)e->cfg.max_games * sizeof(long long)));
    }
    if (pin) {
        // page-lock the caller's arrays so that the copies run at full speed and asynchronously
        cudaError_t err = cudaHostRegister(h_states, (size_t)cap_samples * row * sizeof(float), cudaHostRegisterDefault);
        if (err == cudaSuccess) err = cudaHostRegister(h_distributions, (size_t)cap_samples * A * sizeof(float), cudaHostRegisterDefault);
        if (err == cudaSuccess) err = cudaHostRegister(h_outcomes, (size_t)cap_samples * sizeof(float), cudaHostRegisterDefault);
        if (err != cudaSuccess) {
            cudaGetLastError();
            cudaHostUnregister(h_states); cudaHostUnregister(h_distributions);
            cudaGetLastError();
            return fail(SPRL_E_CAPACITY, "cudaHostRegister of the sample arrays failed: %s", cudaGetErrorString(err));
        }
        so.registered = true;
    }
    so.h_states = h_states; so.h_dists = h_distributions; so.h_outcomes = h_outcomes; so.cap = cap_samples;
    so.games_done = so.rows_done = 0; so.overflow = false; so.which = 0;
    so.active = true;
    return SPRL_OK;
}

int sprl_stream_info(sprl_engine* e, int64_t* games_done, int64_t* samples_done, uint64_t* chunks_while_playing) {
    ENGINE_CHECK(e);
    if (games_done) *games_done = e->so.games_done;
    if (samples_done) *samples_done = e->so.rows_done;
    if (chunks_while_playing) *chunks_while_playing = e->so.chunks;
    return SPRL_OK;
}

int sprl_round(sprl_engine* e) {
    NvtxRange nvtx_range("sprl_round");
    ENGINE_CHECK(e);
    if (!e->iteration_open) return fail(SPRL_E_STATE, "no iteration in progress");
    if (e->cfg.evaluator == SPRL_EVAL_EXTERNAL && !e->p.nn_in) return fail(SPRL_E_STATE, "evaluator buffers are not bound");
    if (e->match_open) {
        search_launch_match_round(e->cfg.game, e->p, e->match, e->stream);
        e->launches += 2;               // the search kernel and the row-counter flip
        ENGINE_CUDA(e, cudaGetLastError());
        return SPRL_OK;
    }
    search_launch_round(e->cfg.game, e->p, e->stream);
    e->launches += 2;               // the search kernel and the order flip
    ENGINE_CUDA(e, cudaGetLastError());
    return SPRL_OK;
}

int sprl_poll(sprl_engine* e, int64_t* slots_playing, int64_t* slots_failed) {
    NvtxRange nvtx_range("sprl_poll");
    ENGINE_CHECK(e);
    unsigned long long c[4] = { 0, 0, 0, 0 };
    ENGINE_CUDA(e, cudaMemcpyAsync(c, e->p.counters, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    if (slots_playing) *slots_playing = e->active_slots - (int64_t)c[0] - (int64_t)c[1];
    if (slots_failed) *slots_failed = (int64_t)c[1];
    if (e->so.active && e->iteration_open && !e->match_open && !e->stepwise && c[1] == 0) {
        const uint64_t before = e->so.games_done;
        int rc = stream_out_advance(e);
        if (rc) return rc;
        if ((uint64_t)e->so.games_done > before && (int64_t)c[0] + (int64_t)c[1] < e->active_slots) e->so.chunks += 1;
    }
    return SPRL_OK;
}

static int report_slot_failure(sprl_engine* e) {
    std::vector<TreeState> ts(e->cfg.num_slots);
    cudaMemcpy(ts.data(), e->p.trees, ts.size() * sizeof(TreeState), cudaMemcpyDeviceToHost);
    for (size_t i = 0; i < ts.size(); ++i) {
        if (ts[i].status == ST_ERR_CAPACITY)
            return fail(SPRL_E_CAPACITY, "tree slot %zu ran out of node units (units_per_tree=%llu, game %llu move %d); raise units_per_tree",
                        i, (unsigned long long)e->p.cap_units, (unsigned long long)ts[i].game_id, ts[i].move_count);
        if (ts[i].status == ST_ERR_ACTION)
            return fail(SPRL_E_INVALID, "tree %zu: the action passed to sprl_advance is not legal at its decision node (or the tree still has leaves waiting for the evaluator)", i);
        if (ts[i].status == ST_ERR_MOVES)
            return fail(SPRL_E_CAPACITY, "tree slot %zu exceeded %d moves in one game", i, e->p.max_moves);
    }
    return fail(SPRL_E_STATE, "a slot failed for an unknown reason");
}

static int run_rounds(sprl_engine* e, bool external, sprl_forward_fn forward, void* user) {
    const int check_every = external ? 64 : 4;
    for (;;) {
        for (int i = 0; i < check_every; ++i) {
            int rc = sprl_round(e);
            if (rc) return rc;
            if (external) {
                rc = forward(user, e->p.nn_in, sprl_eval_batch(e), const_cast<float*>(e->p.nn_logits),
                             const_cast<float*>(e->p.nn_value), (void*)e->stream);
                if (rc) return fail(SPRL_E_STATE, "forward callback returned %d", rc);
            }
        }
        int64_t playing = 0, failed = 0;
        int rc = sprl_poll(e, &playing, &failed);
        if (rc) return rc;
        if (failed > 0) return report_slot_failure(e);
        if (playing == 0) break;
    }
    return SPRL_OK;
}

int sprl_run_iteration(sprl_engine* e, uint64_t first_game, int64_t num_games, sprl_forward_fn forward, void* user) {
    NvtxRange nvtx_range("sprl_run_iteration");
    ENGINE_CHECK(e);
    if (e->cfg.evaluator == SPRL_EVAL_EXTERNAL && !forward) return fail(SPRL_E_INVALID, "SPRL_EVAL_EXTERNAL needs a forward callback");
    int rc = sprl_begin_iteration(e, first_game, num_games);
    if (rc) return rc;
    return run_rounds(e, e->cfg.evaluator == SPRL_EVAL_EXTERNAL, forward, user);
}

int sprl_run_match(sprl_engine* e, const sprl_agent_config* h_agents, uint64_t first_game, int64_t num_games,
                   sprl_forward_fn forward, void* user) {
    NvtxRange nvtx_range("sprl_run_match");
    ENGINE_CHECK(e);
    if (!h_agents) return fail(SPRL_E_INVALID, "null agents");
    const bool external = h_agents[0].evaluator == SPRL_EVAL_EXTERNAL || h_agents[1].evaluator == SPRL_EVAL_EXTERNAL;
    if (external && !forward) return fail(SPRL_E_INVALID, "SPRL_EVAL_EXTERNAL needs a forward callback");
    int rc = sprl_match_begin(e, h_agents, first_game, num_games);
    if (rc) return rc;
    return run_rounds(e, external, forward, user);
}

static int load_game_moves(sprl_engine* e, int64_t* n_moves) {
    e->h_moves.resize((size_t)e->num_games);
    ENGINE_CUDA(e, cudaMemcpyAsync(e->h_moves.data(), e->p.rec_moves, (size_t)e->num_games * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    int64_t total = 0;
    for (int m : e->h_moves) total += m;
    *n_moves = total;
    return SPRL_OK;
}

int sprl_iteration_counts(sprl_engine* e, int64_t* n_moves, int64_t* n_samples) {
    ENGINE_CHECK(e);
    if (!e->iteration_open) return fail(SPRL_E_STATE, "no iteration has been run");
    int64_t moves = 0;
    int rc = load_game_moves(e, &moves);
    if (rc) return rc;
    int S = e->cfg.use_sym ? e->gi.nsym : 1;
    if (n_moves) *n_moves = moves;
    if (n_samples) *n_samples = moves * S;
    return SPRL_OK;
}

int sprl_collect_samples_device(sprl_engine* e, float** d_states, float** d_distributions, float** d_outcomes, int64_t* n_samples) {
    NvtxRange nvtx_range("sprl_collect_samples_device");
    ENGINE_CHECK(e);
    if (!e->iteration_open) return fail(SPRL_E_STATE, "no iteration has been run");
    int64_t moves = 0;
    int rc = load_game_moves(e, &moves);
    if (rc) return rc;
    const int S = e->cfg.use_sym ? e->gi.nsym : 1;
    const int64_t n = moves * S;
    const size_t row = (size_t)(2 * e->gi.history + 1) * e->gi.cells;
    if (n > e->sample_cap || !e->d_row0) {
        if (e->d_states) cudaFree(e->d_states);
        if (e->d_dists) cudaFree(e->d_dists);
        if (e->d_outcomes) cudaFree(e->d_outcomes);
        if (e->d_row0) cudaFree(e->d_row0);
        e->d_states = e->d_dists = e->d_outcomes = nullptr; e->d_row0 = nullptr;
        int64_t cap = std::max<int64_t>(n, 1);
        ENGINE_CUDA(e, cudaMalloc((void**)&e->d_states, (size_t)cap * row * sizeof(float)));
        ENGINE_CUDA(e, cudaMalloc((void**)&e->d_dists, (size_t)cap * e->gi.actions * sizeof(float)));
        ENGINE_CUDA(e, cudaMalloc((void**)&e->d_outcomes, (size_t)cap * sizeof(float)));
        ENGINE_CUDA(e, cudaMalloc((void**)&e->d_row0, (size_t)e->cfg.max_games * sizeof(long long)));
        e->sample_cap = cap;
    }
    std::vector<long long> row0((size_t)e->num_games);
    long long at = 0;
    for (int64_t g = 0; g < e->num_games; ++g) { row0[g] = at; at += (long long)e->h_moves[g] * S; }
    ENGINE_CUDA(e, cudaMemcpyAsync(e->d_row0, row0.data(), row0.size() * sizeof(long long), cudaMemcpyHostToDevice, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));      // row0 is a stack-lifetime host buffer
    if (n > 0) {
        search_launch_emit(e->cfg.game, e->p, 0, e->num_games, e->d_row0, S, e->d_states, e->d_dists, e->d_outcomes, e->stream);
        e->launches += 1;
        ENGINE_CUDA(e, cudaGetLastError());
    }
    if (d_states) *d_states = e->d_states;
    if (d_distributions) *d_distributions = e->d_dists;
    if (d_outcomes) *d_outcomes = e->d_outcomes;
    if (n_samples) *n_samples = n;
    return SPRL_OK;
}

int sprl_collect_samples(sprl_engine* e, int64_t cap_samples, float* h_states, float* h_distributions, float* h_outcomes,
                         int64_t* n_samples) {
    NvtxRange nvtx_range("sprl_collect_samples");
    if (e && e->so.active && h_states == e->so.h_states && h_distributions == e->so.h_dists && h_outcomes == e->so.h_outcomes) {
        // streamed output: most rows are on the host already; embed and copy the games that finished last
        ENGINE_CHECK(e);
        if (!e->iteration_open) return fail(SPRL_E_STATE, "no iteration has been run");
        ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
        int rc = stream_out_advance(e);
        if (rc) return rc;
        for (int k = 0; k < 2; ++k) ENGINE_CUDA(e, cudaStreamSynchronize(e->so.stream[k]));
        int64_t moves = 0;
        for (int m : e->h_moves) moves += m;
        const int64_t total = moves * (e->cfg.use_sym ? e->gi.nsym : 1);
        if (n_samples) *n_samples = total;
        if (e->so.overflow || total > cap_samples || e->so.rows_done != total)
            return fail(SPRL_E_CAPACITY, "%lld samples do not fit the caller's capacity %lld", (long long)total, (long long)std::min(cap_samples, e->so.cap));
        return SPRL_OK;
    }
    int64_t n = 0;
    float *ds, *dd, *dout;
    int rc = sprl_collect_samples_device(e, &ds, &dd, &dout, &n);
    if (rc) return rc;
    if (n_samples) *n_samples = n;
    if (n > cap_samples) return fail(SPRL_E_CAPACITY, "%lld samples do not fit the caller's capacity %lld", (long long)n, (long long)cap_samples);
    const size_t row = (size_t)(2 * e->gi.history + 1) * e->gi.cells;
    if (n > 0) {
        if (h_states) ENGINE_CUDA(e, cudaMemcpyAsync(h_states, ds, (size_t)n * row * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        if (h_distributions) ENGINE_CUDA(e, cudaMemcpyAsync(h_distributions, dd, (size_t)n * e->gi.actions * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        if (h_outcomes) ENGINE_CUDA(e, cudaMemcpyAsync(h_outcomes, dout, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    }
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    return SPRL_OK;
}

int sprl_move_stats(sprl_engine* e, int64_t cap_moves, float* h_N, float* h_W, float* h_P, float* h_root_N,
                    float* h_root_W, int32_t* h_action, int32_t* h_traversals, int8_t* h_player,
                    int32_t* h_game_moves, uint64_t* h_game_draws, int64_t* n_moves) {
    NvtxRange nvtx_range("sprl_move_stats");
    ENGINE_CHECK(e);
    if (!e->cfg.record_stats) return fail(SPRL_E_STATE, "engine was created without record_stats");
    if (!e->iteration_open) return fail(SPRL_E_STATE, "no iteration has been run");
    int64_t moves = 0;
    int rc = load_game_moves(e, &moves);
    if (rc) return rc;
    if (n_moves) *n_moves = moves;
    if (moves > cap_moves) return fail(SPRL_E_CAPACITY, "%lld moves do not fit the caller's capacity %lld", (long long)moves, (long long)cap_moves);
    const size_t A = (size_t)e->gi.actions, MM = (size_t)e->p.max_moves;
    std::vector<int> open((size_t)e->num_games);         // a game's searched moves are recorded after its opening's plies
    ENGINE_CUDA(e, cudaMemcpyAsync(open.data(), e->p.rec_open, open.size() * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    int64_t at = 0;
    for (int64_t g = 0; g < e->num_games; ++g) {
        size_t m = (size_t)e->h_moves[g], src = (size_t)g * MM + (size_t)open[g];
        if (m == 0) continue;
        if (h_N) ENGINE_CUDA(e, cudaMemcpyAsync(h_N + at * A, e->p.rec_N + src * A, m * A * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_W) ENGINE_CUDA(e, cudaMemcpyAsync(h_W + at * A, e->p.rec_W + src * A, m * A * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_P) ENGINE_CUDA(e, cudaMemcpyAsync(h_P + at * A, e->p.rec_P + src * A, m * A * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_root_N) ENGINE_CUDA(e, cudaMemcpyAsync(h_root_N + at, e->p.rec_root_N + src, m * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_root_W) ENGINE_CUDA(e, cudaMemcpyAsync(h_root_W + at, e->p.rec_root_W + src, m * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_action) ENGINE_CUDA(e, cudaMemcpyAsync(h_action + at, e->p.rec_action + src, m * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_traversals) ENGINE_CUDA(e, cudaMemcpyAsync(h_traversals + at, e->p.rec_trav + src, m * 4, cudaMemcpyDeviceToHost, e->stream));
        if (h_player) ENGINE_CUDA(e, cudaMemcpyAsync(h_player + at, e->p.rec_player + src, m, cudaMemcpyDeviceToHost, e->stream));
        at += (int64_t)m;
    }
    if (h_game_moves) memcpy(h_game_moves, e->h_moves.data(), (size_t)e->num_games * sizeof(int));
    if (h_game_draws) ENGINE_CUDA(e, cudaMemcpyAsync(h_game_draws, e->p.rec_draws, (size_t)e->num_games * 8, cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    return SPRL_OK;
}

int sprl_begin_trees(sprl_engine* e, uint64_t first_game, int64_t num_trees) {
    ENGINE_CHECK(e);
    if (num_trees <= 0 || num_trees > e->cfg.num_slots) return fail(SPRL_E_INVALID, "num_trees must be in 1..num_slots (%d)", e->cfg.num_slots);
    e->stepwise = false;
    int rc = sprl_begin_iteration(e, first_game, num_trees);      // one game per tree, started at the start position
    if (rc) return rc;
    e->stepwise = true;
    e->step_sims = 0;
    e->step_single = false;
    return push_iter_params(e);
}

static int stepwise_check(sprl_engine* e) {
    if (!e->iteration_open || !e->stepwise) return fail(SPRL_E_STATE, "no step-wise trees: call sprl_begin_trees first");
    return SPRL_OK;
}

// runs launches until no tree searched or waited for evaluations in the last one
static int stepwise_rounds(sprl_engine* e, sprl_forward_fn forward, void* user, int max_launches) {
    const bool external = e->cfg.evaluator == SPRL_EVAL_EXTERNAL;
    if (external && !forward) return fail(SPRL_E_INVALID, "SPRL_EVAL_EXTERNAL needs a forward callback");
    int rc = push_iter_params(e);
    if (rc) return rc;
    for (int done = 0; max_launches <= 0 || done < max_launches;) {
        const int group = max_launches > 0 ? max_launches - done : 8;
        for (int i = 0; i < group; ++i, ++done) {
            rc = sprl_round(e);
            if (rc) return rc;
            if (external) {
                rc = forward(user, e->p.nn_in, sprl_eval_batch(e), const_cast<float*>(e->p.nn_logits), const_cast<float*>(e->p.nn_value), (void*)e->stream);
                if (rc) return fail(SPRL_E_STATE, "forward callback returned %d", rc);
            }
        }
        unsigned long long c[4] = { 0, 0, 0, 0 };
        ENGINE_CUDA(e, cudaMemcpyAsync(c, e->p.counters, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
        ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
        if (c[1] > 0) return report_slot_failure(e);
        if (c[3] == 0) break;
    }
    return SPRL_OK;
}

int sprl_search(sprl_engine* e, int sims, sprl_forward_fn forward, void* user) {
    NvtxRange nvtx_range("sprl_search");
    ENGINE_CHECK(e);
    int rc = stepwise_check(e);
    if (rc) return rc;
    if (sims < 0) return fail(SPRL_E_INVALID, "sims must not be negative");
    e->step_sims = sims;
    e->step_single = false;
    return stepwise_rounds(e, forward, user, 0);
}

int sprl_search_batch(sprl_engine* e) {
    ENGINE_CHECK(e);
    int rc = stepwise_check(e);
    if (rc) return rc;
    e->step_sims = 0x7fffffff;
    e->step_single = true;
    rc = push_iter_params(e);
    if (!rc) rc = sprl_round(e);
    return rc;
}

int sprl_apply_evaluations(sprl_engine* e) {
    ENGINE_CHECK(e);
    int rc = stepwise_check(e);
    if (rc) return rc;
    e->step_sims = 0;               // every tree only applies what is queued, then waits
    e->step_single = true;
    rc = push_iter_params(e);
    if (!rc) rc = sprl_round(e);
    return rc;
}

int sprl_root_stats(sprl_engine* e, int64_t cap_trees, float* h_N, float* h_W, float* h_P, float* h_root_N, float* h_root_W,
                    int8_t* h_player, int8_t* h_terminal, int8_t* h_winner, int32_t* h_traversals, int8_t* h_mask, int32_t* h_queued) {
    NvtxRange nvtx_range("sprl_root_stats");
    ENGINE_CHECK(e);
    int rc = stepwise_check(e);
    if (rc) return rc;
    const int64_t n = e->num_games;
    if (cap_trees < n) return fail(SPRL_E_CAPACITY, "%lld trees do not fit the caller's capacity %lld", (long long)n, (long long)cap_trees);
    const size_t A = (size_t)e->gi.actions, S = (size_t)e->cfg.num_slots;
    // staging: N, W, P [S][A] floats | root_N, root_W [S] floats | traversals [S] ints | player, terminal, winner [S] | mask [S][A]
    const size_t bytes = 3 * S * A * 4 + 4 * S * 4 + 3 * S + S * A;
    if (!e->d_tree_io) {
        ENGINE_CUDA(e, cudaMalloc((void**)&e->d_tree_io, std::max(bytes, S * sizeof(int))));
        e->allocations.push_back(e->d_tree_io);
    }
    float* dN = (float*)e->d_tree_io; float* dW = dN + S * A; float* dP = dW + S * A;
    float* drn = dP + S * A; float* drw = drn + S;
    int* dtr = (int*)(drw + S);
    int* dqu = dtr + S;
    signed char* dpl = (signed char*)(dqu + S); signed char* dte = dpl + S; signed char* dwi = dte + S; signed char* dmk = dwi + S;
    search_launch_tree_stats(e->cfg.game, e->p, (int)n, dN, dW, dP, drn, drw, dpl, dte, dwi, dtr, dmk, dqu, e->stream);
    e->launches += 1;
    ENGINE_CUDA(e, cudaGetLastError());
    if (h_N) ENGINE_CUDA(e, cudaMemcpyAsync(h_N, dN, (size_t)n * A * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_W) ENGINE_CUDA(e, cudaMemcpyAsync(h_W, dW, (size_t)n * A * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_P) ENGINE_CUDA(e, cudaMemcpyAsync(h_P, dP, (size_t)n * A * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_root_N) ENGINE_CUDA(e, cudaMemcpyAsync(h_root_N, drn, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_root_W) ENGINE_CUDA(e, cudaMemcpyAsync(h_root_W, drw, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_traversals) ENGINE_CUDA(e, cudaMemcpyAsync(h_traversals, dtr, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_queued) ENGINE_CUDA(e, cudaMemcpyAsync(h_queued, dqu, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (h_player) ENGINE_CUDA(e, cudaMemcpyAsync(h_player, dpl, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    if (h_terminal) ENGINE_CUDA(e, cudaMemcpyAsync(h_terminal, dte, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    if (h_winner) ENGINE_CUDA(e, cudaMemcpyAsync(h_winner, dwi, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    if (h_mask) ENGINE_CUDA(e, cudaMemcpyAsync(h_mask, dmk, (size_t)n * A, cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    return SPRL_OK;
}

int sprl_advance(sprl_engine* e, const int32_t* h_actions, int64_t n_actions) {
    NvtxRange nvtx_range("sprl_advance");
    ENGINE_CHECK(e);
    int rc = stepwise_check(e);
    if (rc) return rc;
    if (!h_actions || n_actions != e->num_games) return fail(SPRL_E_INVALID, "sprl_advance takes one action per tree (%lld)", (long long)e->num_games);
    const size_t S = (size_t)e->cfg.num_slots, A = (size_t)e->gi.actions;
    if (!e->d_tree_io) {
        ENGINE_CUDA(e, cudaMalloc((void**)&e->d_tree_io, 3 * S * A * 4 + 4 * S * 4 + 3 * S + S * A));
        e->allocations.push_back(e->d_tree_io);
    }
    ENGINE_CUDA(e, cudaMemcpyAsync(e->d_tree_io, h_actions, (size_t)n_actions * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
    search_launch_tree_advance(e->cfg.game, e->p, (int)n_actions, (const int*)e->d_tree_io, e->stream);
    e->launches += 1;
    ENGINE_CUDA(e, cudaGetLastError());
    unsigned long long c[4] = { 0, 0, 0, 0 };
    ENGINE_CUDA(e, cudaMemcpyAsync(c, e->p.counters, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
    ENGINE_CUDA(e, cudaStreamSynchronize(e->stream));
    if (c[1] > 0) return report_slot_failure(e);
    return SPRL_OK;
}

int sprl_debug_check_guards(sprl_engine* e, int64_t* pools_checked, int64_t* pools_damaged) {
    ENGINE_CHECK(e);
    ENGINE_CUDA(e, cudaDeviceSynchronize());
    int64_t bad = 0;
    std::vector<unsigned char> g(2 * sprl_engine::GUARD);
    for (const sprl_engine::Pool& pl : e->pools) {
        ENGINE_CUDA(e, cudaMemcpy(g.data(), pl.base, sprl_engine::GUARD, cudaMemcpyDeviceToHost));
        ENGINE_CUDA(e, cudaMemcpy(g.data() + sprl_engine::GUARD, pl.base + sprl_engine::GUARD + pl.bytes, sprl_engine::GUARD, cudaMemcpyDeviceToHost));
        bool ok = true;
        for (unsigned char c : g) ok = ok && c == 0xA5;
        if (!ok) ++bad;
    }
    if (pools_checked) *pools_checked = (int64_t)e->pools.size();
    if (pools_damaged) *pools_damaged = bad;
    return SPRL_OK;
}

int sprl_get_stats(sprl_engine* e, sprl_stats* out) {
    ENGINE_CHECK(e);
    if (!out) return fail(SPRL_E_INVALID, "null output");
    sprl_stats now;
    int rc = sum_tree_stats(e, &now);
    if (rc) return rc;
    *out = now;
    out->sims -= e->base.sims; out->evals -= e->base.evals; out->moves -= e->base.moves; out->games -= e->base.games;
    out->depth_sum -= e->base.depth_sum; out->legal_sum -= e->base.legal_sum; out->nodes_visited -= e->base.nodes_visited;
    out->leaves_terminal -= e->base.leaves_terminal; out->leaves_gray -= e->base.leaves_gray; out->leaves_empty -= e->base.leaves_empty;
    out->leaves_duplicate -= e->base.leaves_duplicate;
    out->launches -= e->base.launches;
    return SPRL_OK;
}

int sprl_reset_stats(sprl_engine* e) {
    ENGINE_CHECK(e);
    return sum_tree_stats(e, &e->base);
}

int sprl_write_npy_f32(const char* path, const float* h_data, const uint64_t* shape, int ndim) {
    if (!path || (!h_data && ndim > 0) || ndim < 0 || ndim > 8) return fail(SPRL_E_INVALID, "bad argument to sprl_write_npy_f32");
    // utils/npy.hpp:430-476: v1.0 header, dict padded with spaces to a multiple of 16 (a full 16 when already aligned)
    std::string tuple;
    uint64_t count = 1;
    if (ndim == 0) tuple = "()";
    else if (ndim == 1) tuple = "(" + std::to_string(shape[0]) + ",)";
    else {
        tuple = "(";
        for (int i = 0; i < ndim; ++i) tuple += std::to_string(shape[i]) + (i + 1 < ndim ? ", " : ")");
    }
    for (int i = 0; i < ndim; ++i) count *= shape[i];
    std::string dict = "{'descr': '<f4', 'fortran_order': False, 'shape': " + tuple + ", }";
    size_t length = 6 + 2 + 2 + dict.size() + 1;
    size_t pad = 16 - length % 16;
    size_t hlen = dict.size() + pad + 1;
    if (hlen > 65535) return fail(SPRL_E_INVALID, "npy header too long");
    FILE* f = fopen(path, "wb");
    if (!f) return fail(SPRL_E_IO, "io error: failed to open %s", path);
    const unsigned char magic[10] = { 0x93, 'N', 'U', 'M', 'P', 'Y', 1, 0, (unsigned char)(hlen & 0xff), (unsigned char)(hlen >> 8) };
    bool ok = fwrite(magic, 1, 10, f) == 10 && fwrite(dict.data(), 1, dict.size(), f) == dict.size();
    std::string padding(pad, ' ');
    padding += '\n';
    ok = ok && fwrite(padding.data(), 1, padding.size(), f) == padding.size();
    ok = ok && (count == 0 || fwrite(h_data, sizeof(float), (size_t)count, f) == (size_t)count);
    ok = (fclose(f) == 0) && ok;
    if (!ok) return fail(SPRL_E_IO, "io error: short write to %s", path);
    return SPRL_OK;
}

}  // extern "C"
