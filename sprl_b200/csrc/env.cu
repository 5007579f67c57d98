// env.cu -- environment-only kernels (BASELINE config 2): batched transitions,
// random playouts and breadth-first perft over the bitboard rules of games.cuh.
// Replaces, for many positions at once, GameNode::getAddChild and the accessors of
// /root/reference/cpp/src/games/GameNode.hpp:96-160.
#include <vector>

#include "common.cuh"
#include "games.cuh"
#include "rng.cuh"

namespace sprl {

thread_local std::string g_last_error;
std::string& last_error_ref() { return g_last_error; }

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

int use_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(SPRL_E_NOGPU, "no CUDA device available (%s); libsprl_b200 has no CPU path",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= n) return fail(SPRL_E_INVALID, "device %d out of range (have %d)", device, n);
    SPRL_CUDA(cudaSetDevice(device));
    return SPRL_OK;
}

// History of the boards of one line of play, oldest first: [count][2*W] words.
template <int W>
struct LineHist {
    const u64* data;
    int count;
    __host__ __device__ bool seen(const Bits<W>& b0, const Bits<W>& b1) const {
        for (int i = 0; i < count; ++i) {
            bool same = true;
            for (int w = 0; w < W; ++w)
                same = same && data[(size_t)i * 2 * W + w] == b0.word(w) && data[(size_t)i * 2 * W + W + w] == b1.word(w);
            if (same) return true;
        }
        return false;
    }
    template <class F> __host__ __device__ void for_each(F&& f) const {
        for (int i = 0; i < count; ++i) {
            Bits<W> b0, b1;
            for (int w = 0; w < W; ++w) { b0.set_word(w, data[(size_t)i * 2 * W + w]); b1.set_word(w, data[(size_t)i * 2 * W + W + w]); }
            f(b0, b1);
        }
    }
};

// ---- batched single transitions ----------------------------------------------------
template <class G>
__global__ void k_env_step(int64_t n, const u64* __restrict__ b0, const u64* __restrict__ b1,
                           const unsigned char* __restrict__ player, const int* __restrict__ action,
                           PosRec* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    typename G::P par, nx;
    par.b[0] = Bits<1>(b0[i]); par.b[1] = Bits<1>(b1[i]);
    par.player = player[i]; par.depth = 0; par.action = 0; par.terminal = 0; par.winner = WINNER_NONE;
    par.pass_legal = 0;
    G::next(par, action[i], NoHistory(), nx);
    pos_to_rec<G>(nx, out[i]);
}

// ---- lines of play from the start position (chains of GameNode::getAddChild calls, games/GameNode.hpp:96-110) ----
// One thread per line: a line is sequential.  Line i = actions[off[i] .. off[i+1]-1]; rec[off[i] + i + k] = the position
// after k of its actions, k = 0 .. its length (rec_to_pos restores each exactly, depth included); for Go the line is the
// history of the positional-superko rule, kept in hist[off[i] ..].  bad[i] = index of the first action of line i that is
// not legal where it is played (or -1).
template <class G>
__global__ void k_env_lines(int n_lines, const long long* __restrict__ off, const int* __restrict__ actions,
                            PosRec* __restrict__ rec, u64* __restrict__ hist /* [total actions][2W] */, int* __restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lines) return;
    const long long a0 = off[i];
    const int n_actions = (int)(off[i + 1] - a0);
    const int* act = actions + a0;
    PosRec* r = rec + a0 + i;
    u64* h = hist + (size_t)a0 * 2 * G::W;
    typename G::P cur, nx;
    G::start(cur);
    bad[i] = -1;
    for (int k = 0;; ++k) {
        pos_to_rec<G>(cur, r[k]);
        if (k == n_actions) break;
        const int a = act[k];
        const bool legal = !cur.terminal && a >= 0 && a < G::ACTIONS &&
                           ((G::HAS_PASS && a == G::CELLS) ? cur.pass_legal != 0 : cur.legal.test(a));
        if (!legal) { bad[i] = k; break; }
        const LineHist<G::W> lh = { h, k };                 // the positions before `cur`; next() adds `cur` and the new one
        G::next(cur, a, lh, nx);
        for (int w = 0; w < G::W; ++w) {
            h[(size_t)k * 2 * G::W + w] = cur.b[0].word(w);
            h[(size_t)k * 2 * G::W + G::W + w] = cur.b[1].word(w);
        }
        cur = nx;
    }
}

void env_launch_lines(int game, int n_lines, const long long* off, const int* actions, PosRec* rec, u64* hist, int* bad,
                      cudaStream_t s) {
    const int grid = ceil_div(n_lines, 128);
    switch (game) {
    case SPRL_GAME_OTHELLO: k_env_lines<Othello><<<grid, 128, 0, s>>>(n_lines, off, actions, rec, hist, bad); break;
    case SPRL_GAME_C4: k_env_lines<ConnectFour><<<grid, 128, 0, s>>>(n_lines, off, actions, rec, hist, bad); break;
    case SPRL_GAME_GO7: k_env_lines<Go<7>><<<grid, 128, 0, s>>>(n_lines, off, actions, rec, hist, bad); break;
    case SPRL_GAME_GO9: k_env_lines<Go<9>><<<grid, 128, 0, s>>>(n_lines, off, actions, rec, hist, bad); break;
    default: break;
    }
}

// ---- random playouts, one thread per game ----------------------------------------------
template <class G>
__global__ void k_rollout(uint64_t seed, uint64_t first_game, int64_t ngames, int max_steps,
                          int* __restrict__ game_steps, unsigned char* __restrict__ final_winner,
                          PosRec* __restrict__ rec /* [ngames, max_steps] or null */,
                          u64* __restrict__ hist /* Go: [ngames, max_steps, 2W] */,
                          unsigned long long* __restrict__ total_steps) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long my_steps = 0;
    if (g < ngames) {
        Rng rng = { seed, first_game + (uint64_t)g, 0 };
        typename G::P cur, nx;
        G::start(cur);
        u64* myhist = hist ? hist + (size_t)g * max_steps * 2 * G::W : nullptr;
        int steps = 0;
        for (;;) {
            int n = cur.n_legal();
            int pick = -1;
            if (!cur.terminal) pick = legal_action<G>(cur, rng_uniform_int(rng, 0, n - 1));
            if (rec) {
                PosRec r;
                pos_to_rec<G>(cur, r);
                r.action = pick;
                rec[(size_t)g * max_steps + steps] = r;
            }
            ++steps;
            if (cur.terminal) break;
            if (myhist) {
                LineHist<G::W> lh = { myhist, steps - 1 };
                G::next(cur, pick, lh, nx);
                for (int w = 0; w < G::W; ++w) {
                    myhist[(size_t)(steps - 1) * 2 * G::W + w] = cur.b[0].word(w);
                    myhist[(size_t)(steps - 1) * 2 * G::W + G::W + w] = cur.b[1].word(w);
                }
            } else {
                G::next(cur, pick, NoHistory(), nx);
            }
            cur = nx;
        }
        game_steps[g] = steps;
        final_winner[g] = cur.winner;
        my_steps = (unsigned long long)(steps - 1);
    }
    // one atomic per warp
    for (int o = 16; o > 0; o >>= 1) my_steps += __shfl_down_sync(0xffffffffu, my_steps, o);
    if ((threadIdx.x & 31) == 0 && my_steps) atomicAdd(total_steps, my_steps);
}

// ---- perft: breadth-first frontier expansion -------------------------------------------
struct PerftLevels {
    const PosRec* level[40];
};

// walks the parents of a frontier entry through the stored levels
template <int W>
struct PerftHist {
    const PerftLevels* lv;
    int depth;      // level of the parent entry
    u32 index;      // index of the parent entry within its level
    __device__ bool seen(const Bits<W>& b0, const Bits<W>& b1) const {
        // strict ancestors of the parent entry
        int d = depth;
        u32 idx = index;
        while (d > 0) {
            idx = lv->level[d][idx].parent;
            --d;
            const PosRec& r = lv->level[d][idx];
            bool same = true;
            for (int w = 0; w < W; ++w) same = same && r.b[w] == b0.word(w) && r.b[2 + w] == b1.word(w);
            if (same) return true;
        }
        return false;
    }
    template <class F> __device__ void for_each(F&& f) const {
        int d = depth;
        u32 idx = index;
        while (d > 0) {
            idx = lv->level[d][idx].parent;
            --d;
            const PosRec& r = lv->level[d][idx];
            Bits<W> b0, b1;
            for (int w = 0; w < W; ++w) { b0.set_word(w, r.b[w]); b1.set_word(w, r.b[2 + w]); }
            f(b0, b1);
        }
    }
};

template <class G>
__global__ void k_perft_count(const PosRec* __restrict__ level, int64_t n,
                              unsigned long long* __restrict__ children, unsigned long long* __restrict__ terminals) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long c = 0, t = 0;
    if (i < n) {
        const PosRec& r = level[i];
        if (r.terminal) t = 1;
        else c = (unsigned long long)(__popcll(r.legal[0]) + __popcll(r.legal[1]) + r.pass_legal);
    }
    for (int o = 16; o > 0; o >>= 1) {
        c += __shfl_down_sync(0xffffffffu, c, o);
        t += __shfl_down_sync(0xffffffffu, t, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (c) atomicAdd(children, c);
        if (t) atomicAdd(terminals, t);
    }
}

// One warp expands 32 parents together: the children of the 32 parents are numbered by a warp scan,
// the warp reserves their slots with ONE atomicAdd, and lane j generates child j (its parent found by
// a binary search over the scan), so lanes stay busy whatever the parents' move counts are and
// neighbouring lanes write neighbouring records.
template <class G>
__global__ void k_perft_expand(PerftLevels lv, int depth, int64_t n, PosRec* __restrict__ next,
                               unsigned long long* __restrict__ cursor) {
    constexpr unsigned FULL = 0xffffffffu;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int64_t i0 = i - lane;
    const PosRec* __restrict__ level = lv.level[depth];
    int nl = 0;
    if (i < n) {
        const PosRec& r = level[i];
        if (!r.terminal) nl = __popcll(r.legal[0]) + __popcll(r.legal[1]) + r.pass_legal;
    }
    int incl = nl;
    for (int o = 1; o < 32; o <<= 1) {
        int v = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    if (total == 0) return;
    const int excl = incl - nl;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(cursor, (unsigned long long)total);
    base = __shfl_sync(FULL, base, 0);
    for (int j0 = 0; j0 < total; j0 += 32) {
        const int j = j0 + lane;
        int src = 0;        // last lane whose first child is <= j
        for (int step = 16; step > 0; step >>= 1) {
            const int cand = src + step;
            const int e = __shfl_sync(FULL, excl, cand & 31);
            if (cand < 32 && e <= j) src = cand;
        }
        const int first = __shfl_sync(FULL, excl, src);
        if (j < total) {
            typename G::P par, nx;
            rec_to_pos<G>(level[i0 + src], par);
            PerftHist<G::W> hist = { &lv, depth, (u32)(i0 + src) };
            G::next(par, legal_action<G>(par, j - first), hist, nx);
            PosRec o;
            pos_to_rec<G>(nx, o);
            o.parent = (u32)(i0 + src);
            next[base + j] = o;
        }
    }
}

// ---- host side ---------------------------------------------------------------------------
template <class G>
static void cells_from_rec(const PosRec& r, int8_t* cells) {
    for (int i = 0; i < G::CELLS; ++i) {
        bool z = (r.b[i >> 6] >> (i & 63)) & 1ULL, o = (r.b[2 + (i >> 6)] >> (i & 63)) & 1ULL;
        cells[i] = z ? 0 : (o ? 1 : -1);
    }
}
template <class G>
static void mask_from_rec(const PosRec& r, int8_t* mask) {
    if constexpr (!G::HAS_PASS) {
        for (int a = 0; a < G::ACTIONS; ++a) mask[a] = (r.legal[0] >> a) & 1ULL;
    } else {
        for (int i = 0; i < G::CELLS; ++i) mask[i] = (r.legal[i >> 6] >> (i & 63)) & 1ULL;
        mask[G::CELLS] = r.pass_legal;
    }
}
static int8_t winner_code(unsigned char w) { return w == WINNER_ZERO ? 0 : (w == WINNER_ONE ? 1 : -1); }

template <class G>
static int env_step_impl(int64_t n, const int8_t* h_cells, const int8_t* h_player, const int32_t* h_action,
                         int8_t* h_next_cells, int8_t* h_next_player, int8_t* h_terminal, int8_t* h_winner,
                         int8_t* h_mask) {
    std::vector<u64> b0(n), b1(n);
    std::vector<unsigned char> pl(n);
    for (int64_t i = 0; i < n; ++i) {
        u64 z = 0, o = 0;
        for (int c = 0; c < G::CELLS; ++c) {
            int8_t v = h_cells[i * G::CELLS + c];
            if (v == 0) z |= 1ULL << c; else if (v == 1) o |= 1ULL << c;
        }
        b0[i] = z; b1[i] = o; pl[i] = (unsigned char)h_player[i];
        if (h_action[i] < 0 || h_action[i] >= G::ACTIONS) return fail(SPRL_E_INVALID, "action %d out of range at %lld", h_action[i], (long long)i);
    }
    DeviceBuf<u64> d0, d1; DeviceBuf<unsigned char> dp; DeviceBuf<int> da; DeviceBuf<PosRec> dout;
    SPRL_CUDA(d0.alloc(n)); SPRL_CUDA(d1.alloc(n)); SPRL_CUDA(dp.alloc(n)); SPRL_CUDA(da.alloc(n)); SPRL_CUDA(dout.alloc(n));
    SPRL_CUDA(cudaMemcpy(d0.p, b0.data(), n * 8, cudaMemcpyHostToDevice));
    SPRL_CUDA(cudaMemcpy(d1.p, b1.data(), n * 8, cudaMemcpyHostToDevice));
    SPRL_CUDA(cudaMemcpy(dp.p, pl.data(), n, cudaMemcpyHostToDevice));
    SPRL_CUDA(cudaMemcpy(da.p, h_action, n * 4, cudaMemcpyHostToDevice));
    k_env_step<G><<<ceil_div(n, 256), 256>>>(n, d0.p, d1.p, dp.p, da.p, dout.p);
    SPRL_CUDA(cudaGetLastError());
    std::vector<PosRec> out(n);
    SPRL_CUDA(cudaMemcpy(out.data(), dout.p, n * sizeof(PosRec), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n; ++i) {
        cells_from_rec<G>(out[i], h_next_cells + i * G::CELLS);
        h_next_player[i] = out[i].player;
        h_terminal[i] = out[i].terminal;
        h_winner[i] = winner_code(out[i].winner);
        mask_from_rec<G>(out[i], h_mask + i * G::ACTIONS);
    }
    return SPRL_OK;
}

template <class G>
static int env_rollout_impl(uint64_t seed, uint64_t first_game, int64_t ngames, int32_t* h_game_steps,
                            int8_t* h_final_winner, int64_t cap, int8_t* h_cells, int8_t* h_player,
                            int8_t* h_terminal, int8_t* h_winner, int8_t* h_mask, int32_t* h_action,
                            int64_t* total_positions, float* elapsed_ms) {
    const int max_steps = G::MAX_PLIES + 1;
    const bool record = h_cells != nullptr;
    const bool need_hist = (G::KIND == GAME_GO7 || G::KIND == GAME_GO9);
    DeviceBuf<int> dsteps; DeviceBuf<unsigned char> dwin; DeviceBuf<PosRec> drec; DeviceBuf<u64> dhist;
    DeviceBuf<unsigned long long> dtotal;
    SPRL_CUDA(dsteps.alloc(ngames)); SPRL_CUDA(dwin.alloc(ngames)); SPRL_CUDA(dtotal.alloc(1));
    if (record) SPRL_CUDA(drec.alloc((size_t)ngames * max_steps));
    if (need_hist) SPRL_CUDA(dhist.alloc((size_t)ngames * max_steps * 2 * G::W));
    SPRL_CUDA(cudaMemset(dtotal.p, 0, 8));
    cudaEvent_t e0, e1;
    SPRL_CUDA(cudaEventCreate(&e0)); SPRL_CUDA(cudaEventCreate(&e1));
    SPRL_CUDA(cudaEventRecord(e0));
    k_rollout<G><<<ceil_div(ngames, 128), 128>>>(seed, first_game, ngames, max_steps, dsteps.p, dwin.p,
                                                  record ? drec.p : nullptr, need_hist ? dhist.p : nullptr, dtotal.p);
    SPRL_CUDA(cudaGetLastError());
    SPRL_CUDA(cudaEventRecord(e1));
    SPRL_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    SPRL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (elapsed_ms) *elapsed_ms = ms;
    std::vector<int> steps(ngames);
    std::vector<unsigned char> win(ngames);
    SPRL_CUDA(cudaMemcpy(steps.data(), dsteps.p, ngames * 4, cudaMemcpyDeviceToHost));
    SPRL_CUDA(cudaMemcpy(win.data(), dwin.p, ngames, cudaMemcpyDeviceToHost));
    int64_t total = 0;
    for (int64_t g = 0; g < ngames; ++g) {
        if (h_game_steps) h_game_steps[g] = steps[g];
        if (h_final_winner) h_final_winner[g] = winner_code(win[g]);
        total += steps[g];
    }
    if (total_positions) *total_positions = total;
    if (record) {
        if (total > cap) return fail(SPRL_E_CAPACITY, "rollout trace needs %lld positions, capacity %lld", (long long)total, (long long)cap);
        std::vector<PosRec> rec((size_t)ngames * max_steps);
        SPRL_CUDA(cudaMemcpy(rec.data(), drec.p, rec.size() * sizeof(PosRec), cudaMemcpyDeviceToHost));
        int64_t at = 0;
        for (int64_t g = 0; g < ngames; ++g)
            for (int s = 0; s < steps[g]; ++s, ++at) {
                const PosRec& r = rec[(size_t)g * max_steps + s];
                cells_from_rec<G>(r, h_cells + at * G::CELLS);
                h_player[at] = r.player; h_terminal[at] = r.terminal; h_winner[at] = winner_code(r.winner);
                mask_from_rec<G>(r, h_mask + at * G::ACTIONS);
                h_action[at] = r.action;
            }
    }
    return SPRL_OK;
}

template <class G>
static int env_line_impl(int32_t n_actions, const int32_t* h_actions, int8_t* h_cells, int8_t* h_player, int8_t* h_terminal,
                         int8_t* h_winner, int8_t* h_mask) {
    if (n_actions > G::MAX_PLIES) return fail(SPRL_E_INVALID, "a line of %d actions is longer than a game (%d plies)", n_actions, G::MAX_PLIES);
    const size_t n = (size_t)n_actions + 1;
    const long long off[2] = { 0, n_actions };
    DeviceBuf<int> dact, dbad; DeviceBuf<PosRec> drec; DeviceBuf<u64> dhist; DeviceBuf<long long> doff;
    SPRL_CUDA(dact.alloc(n)); SPRL_CUDA(dbad.alloc(1)); SPRL_CUDA(drec.alloc(n)); SPRL_CUDA(dhist.alloc(n * 2 * G::W));
    SPRL_CUDA(doff.alloc(2));
    SPRL_CUDA(cudaMemcpy(doff.p, off, sizeof(off), cudaMemcpyHostToDevice));
    if (n_actions) SPRL_CUDA(cudaMemcpy(dact.p, h_actions, (size_t)n_actions * 4, cudaMemcpyHostToDevice));
    k_env_lines<G><<<1, 32>>>(1, doff.p, dact.p, drec.p, dhist.p, dbad.p);
    SPRL_CUDA(cudaGetLastError());
    int bad = -1;
    SPRL_CUDA(cudaMemcpy(&bad, dbad.p, 4, cudaMemcpyDeviceToHost));
    if (bad >= 0) return fail(SPRL_E_INVALID, "action %d (index %d of the line) is not legal in the position it is played in", h_actions[bad], bad);
    std::vector<PosRec> rec(n);
    SPRL_CUDA(cudaMemcpy(rec.data(), drec.p, n * sizeof(PosRec), cudaMemcpyDeviceToHost));
    for (size_t k = 0; k < n; ++k) {
        if (h_cells) cells_from_rec<G>(rec[k], h_cells + k * G::CELLS);
        if (h_player) h_player[k] = rec[k].player;
        if (h_terminal) h_terminal[k] = rec[k].terminal;
        if (h_winner) h_winner[k] = winner_code(rec[k].winner);
        if (h_mask) mask_from_rec<G>(rec[k], h_mask + k * G::ACTIONS);
    }
    return SPRL_OK;
}

template <class G>
static int env_perft_impl(int depth, uint64_t* count, float* elapsed_ms) {
    if (depth < 0 || depth >= 40) return fail(SPRL_E_INVALID, "perft depth %d out of range", depth);
    cudaEvent_t e0, e1;
    SPRL_CUDA(cudaEventCreate(&e0)); SPRL_CUDA(cudaEventCreate(&e1));
    std::vector<PosRec*> levels;        // every level stays resident (PerftHist walks the ancestors)
    std::vector<PosRec*> owned;         // separate allocations of levels that did not fit the arena
    // Frontier arena taken before the timed region; 2 GiB holds every level of Othello perft(11).
    PosRec* arena = nullptr;
    size_t arena_recs = depth >= 6 ? ((size_t)2 << 30) / sizeof(PosRec) : (size_t)1 << 16, arena_used = 0;
    if (cudaMalloc((void**)&arena, arena_recs * sizeof(PosRec)) != cudaSuccess) { cudaGetLastError(); arena = nullptr; arena_recs = 0; }
    auto cleanup = [&]() { for (PosRec* p : owned) cudaFree(p); cudaFree(arena); cudaEventDestroy(e0); cudaEventDestroy(e1); };
    PerftLevels lv;
    for (int i = 0; i < 40; ++i) lv.level[i] = nullptr;
    DeviceBuf<unsigned long long> dctr;
    SPRL_CUDA(dctr.alloc(3));
    typename G::P start;
    G::start(start);
    PosRec r0;
    pos_to_rec<G>(start, r0);
    PosRec* d0 = nullptr;
    if (arena_recs) { d0 = arena; arena_used = 1; }
    else {
        if (cudaMalloc((void**)&d0, sizeof(PosRec)) != cudaSuccess) { cleanup(); return fail(SPRL_E_CUDA, "perft: out of device memory"); }
        owned.push_back(d0);
    }
    levels.push_back(d0);
    lv.level[0] = d0;
    cudaError_t err = cudaMemcpy(d0, &r0, sizeof(PosRec), cudaMemcpyHostToDevice);
    if (err != cudaSuccess) { cleanup(); return fail(SPRL_E_CUDA, "perft upload: %s", cudaGetErrorString(err)); }
    cudaEventRecord(e0);
    uint64_t n = 1, terminals_above = 0, result = 0;
    if (depth == 0) result = 1;
    for (int d = 0; d < depth; ++d) {
        unsigned long long h[3] = { 0, 0, 0 };
        cudaMemcpy(dctr.p, h, 24, cudaMemcpyHostToDevice);
        k_perft_count<G><<<ceil_div((long long)n, 256), 256>>>(levels[d], (int64_t)n, dctr.p, dctr.p + 1);
        err = cudaMemcpy(h, dctr.p, 24, cudaMemcpyDeviceToHost);
        if (err != cudaSuccess) { cleanup(); return fail(SPRL_E_CUDA, "perft count at depth %d: %s", d, cudaGetErrorString(err)); }
        terminals_above += h[1];
        if (d == depth - 1) { result = terminals_above + h[0]; break; }
        if (h[0] == 0) { result = terminals_above; break; }
        PosRec* nxt = nullptr;
        if (arena_used + h[0] <= arena_recs) { nxt = arena + arena_used; arena_used += h[0]; }
        else {
            err = cudaMalloc((void**)&nxt, (size_t)h[0] * sizeof(PosRec));
            if (err != cudaSuccess) { cleanup(); return fail(SPRL_E_CAPACITY, "perft frontier of %llu positions: %s", h[0], cudaGetErrorString(err)); }
            owned.push_back(nxt);
        }
        levels.push_back(nxt);
        lv.level[d + 1] = nxt;
        k_perft_expand<G><<<ceil_div((long long)n, 128), 128>>>(lv, d, (int64_t)n, nxt, dctr.p + 2);
        err = cudaGetLastError();
        if (err != cudaSuccess) { cleanup(); return fail(SPRL_E_CUDA, "perft expand at depth %d: %s", d, cudaGetErrorString(err)); }
        n = h[0];
    }
    cudaEventRecord(e1);
    err = cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cleanup();
    if (err != cudaSuccess) return fail(SPRL_E_CUDA, "perft: %s", cudaGetErrorString(err));
    if (elapsed_ms) *elapsed_ms = ms;
    *count = result;
    return SPRL_OK;
}

}  // namespace sprl

using namespace sprl;

#define DISPATCH_GAME(game, CALL)                                                    \
    switch (game) {                                                                  \
    case SPRL_GAME_OTHELLO: { typedef Othello G; return CALL; }                      \
    case SPRL_GAME_C4: { typedef ConnectFour G; return CALL; }                       \
    case SPRL_GAME_GO7: { typedef Go<7> G; return CALL; }                            \
    case SPRL_GAME_GO9: { typedef Go<9> G; return CALL; }                            \
    default: return fail(SPRL_E_INVALID, "unknown game %d", game);                   \
    }

template <class G> static int game_info_impl(sprl_game_info* out) {
    out->rows = G::ROWS; out->cols = G::COLS; out->cells = G::CELLS; out->actions = G::ACTIONS;
    out->history = G::HISTORY; out->nsym = G::NSYM; out->max_plies = G::MAX_PLIES;
    return SPRL_OK;
}

extern "C" {

const char* sprl_last_error(void) { return last_error_ref().c_str(); }

int sprl_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int sprl_game_info_get(int game, sprl_game_info* out) {
    if (!out) return fail(SPRL_E_INVALID, "null output");
    DISPATCH_GAME(game, game_info_impl<G>(out));
}

int sprl_env_step(int device, int game, int64_t n, const int8_t* h_cells, const int8_t* h_player,
                  const int32_t* h_action, int8_t* h_next_cells, int8_t* h_next_player,
                  int8_t* h_terminal, int8_t* h_winner, int8_t* h_mask) {
    NvtxRange nvtx_range("sprl_env_step");
    if (n < 0 || !h_cells || !h_player || !h_action || !h_next_cells || !h_next_player || !h_terminal || !h_winner || !h_mask)
        return fail(SPRL_E_INVALID, "sprl_env_step: null buffer or negative count");
    if (n == 0) return SPRL_OK;
    int rc = use_device(device);
    if (rc) return rc;
    switch (game) {
    case SPRL_GAME_OTHELLO: return env_step_impl<Othello>(n, h_cells, h_player, h_action, h_next_cells, h_next_player, h_terminal, h_winner, h_mask);
    case SPRL_GAME_C4: return env_step_impl<ConnectFour>(n, h_cells, h_player, h_action, h_next_cells, h_next_player, h_terminal, h_winner, h_mask);
    default: return fail(SPRL_E_INVALID, "sprl_env_step supports Othello and Connect Four (game %d needs its history)", game);
    }
}

int sprl_env_line(int device, int game, int32_t n_actions, const int32_t* h_actions, int8_t* h_cells, int8_t* h_player,
                  int8_t* h_terminal, int8_t* h_winner, int8_t* h_mask) {
    NvtxRange nvtx_range("sprl_env_line");
    if (n_actions < 0 || (n_actions > 0 && !h_actions)) return fail(SPRL_E_INVALID, "sprl_env_line: negative length or null actions");
    int rc = use_device(device);
    if (rc) return rc;
    DISPATCH_GAME(game, env_line_impl<G>(n_actions, h_actions, h_cells, h_player, h_terminal, h_winner, h_mask));
}

int sprl_env_rollout(int device, int game, uint64_t seed, uint64_t first_game, int64_t ngames,
                     int32_t* h_game_steps, int8_t* h_final_winner, int64_t cap,
                     int8_t* h_cells, int8_t* h_player, int8_t* h_terminal, int8_t* h_winner,
                     int8_t* h_mask, int32_t* h_action, int64_t* total_positions, float* elapsed_ms) {
    NvtxRange nvtx_range("sprl_env_rollout");
    if (ngames < 0) return fail(SPRL_E_INVALID, "negative game count");
    if (h_cells && (!h_player || !h_terminal || !h_winner || !h_mask || !h_action))
        return fail(SPRL_E_INVALID, "sprl_env_rollout: trace buffers must be given together");
    if (ngames == 0) { if (total_positions) *total_positions = 0; return SPRL_OK; }
    int rc = use_device(device);
    if (rc) return rc;
    DISPATCH_GAME(game, env_rollout_impl<G>(seed, first_game, ngames, h_game_steps, h_final_winner, cap, h_cells,
                                            h_player, h_terminal, h_winner, h_mask, h_action, total_positions, elapsed_ms));
}

int sprl_env_perft(int device, int game, int depth, uint64_t* count, float* elapsed_ms) {
    NvtxRange nvtx_range("sprl_env_perft");
    if (!count) return fail(SPRL_E_INVALID, "null output");
    int rc = use_device(device);
    if (rc) return rc;
    DISPATCH_GAME(game, env_perft_impl<G>(depth, count, elapsed_ms));
}

}  // extern "C"
