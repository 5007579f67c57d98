// search.cu -- warp-per-tree UCT search, move finalisation, subtree compaction and
// sample emission.  Restates on the device, with the reference's fp32 operand
// order, what /root/reference/cpp/src/uct/UCTTree.hpp, uct/UCTNode.hpp and
// selfplay/SelfPlay.hpp do per game; see search.cuh for the data model.
//
// Every branch on tree state below is warp-uniform: all 32 lanes of the owning
// warp hold identical copies of the tree registers and of the RNG stream, and
// only the parts marked "lane k" diverge (one lane per edge / cell).
#include "common.cuh"
#include "search.cuh"

namespace sprl {

#define FULL 0xffffffffu

// ---- symmetries (symmetry/D4GridSymmetrizer.hpp:106-117, ConnectFourSymmetrizer.cpp) ----
template <class G>
__device__ __forceinline__ int sym_cell(int s, int from) {     // to = f_s(from)
    if (G::KIND == GAME_C4) {
        int r = from / 7, c = from - r * 7;
        return s == 1 ? r * 7 + (6 - c) : from;
    }
    // D4 element s = optional transpose, then optional flips of the row / column index:
    // 0 (r,c)  1 (c,w-1-r)  2 (w-1-r,w-1-c)  3 (w-1-c,r)  4 (r,w-1-c)  5 (w-1-c,w-1-r)  6 (w-1-r,c)  7 (c,r)
    const int w = G::COLS;
    const int r = from / w, c = from - r * w;
    const bool swap = (0xAA >> s) & 1, flip_r = (0x6C >> s) & 1, flip_c = (0x36 >> s) & 1;
    const int a = swap ? c : r, b = swap ? r : c;
    const int tr = flip_r ? w - 1 - a : a, tc = flip_c ? w - 1 - b : b;
    return tr * w + tc;
}
template <class G>
__device__ __forceinline__ int sym_action(int s, int a) {
    if (G::KIND == GAME_C4) return s == 1 ? 6 - a : a;
    return a == G::CELLS ? a : sym_cell<G>(s, a);
}
template <class G>
__device__ __forceinline__ int sym_inverse(int s) {             // D4GridSymmetrizer.hpp:47-50
    if (G::KIND == GAME_C4) return s;
    return (s == 1) ? 3 : ((s == 3) ? 1 : s);
}

// ---- node header in registers ---------------------------------------------------------------
template <int W>
struct Hdr {
    Bits<W> b0, b1, legal;
    u32 parent, own_edge;
    float net_value;
    u32 meta, aux;
};

template <int W> struct HL;
template <> struct HL<1> {
    static constexpr int HDR = 3;
    __device__ static void load(const uint4* p, Hdr<1>& h) {
        uint4 a = p[0], b = p[1], c = p[2];
        h.b0 = Bits<1>((u64)a.x | ((u64)a.y << 32));
        h.b1 = Bits<1>((u64)a.z | ((u64)a.w << 32));
        h.legal = Bits<1>((u64)b.x | ((u64)b.y << 32));
        h.parent = b.z; h.own_edge = b.w;
        h.net_value = __uint_as_float(c.x); h.meta = c.y; h.aux = c.z;
    }
    __device__ static void store_unit(uint4* p, int i, const Hdr<1>& h) {
        if (i == 0) p[0] = make_uint4((u32)h.b0.w0, (u32)(h.b0.w0 >> 32), (u32)h.b1.w0, (u32)(h.b1.w0 >> 32));
        else if (i == 1) p[1] = make_uint4((u32)h.legal.w0, (u32)(h.legal.w0 >> 32), h.parent, h.own_edge);
        else p[2] = make_uint4(__float_as_uint(h.net_value), h.meta, h.aux, 0u);
    }
    __device__ static u32* meta_ptr(uint4* p) { return reinterpret_cast<u32*>(p + 2) + 1; }
    __device__ static float* value_ptr(uint4* p) { return reinterpret_cast<float*>(p + 2); }
    // header unit `u` of a record moved by re-rooting: new links, expanded bit cleared
    __device__ static void relink_unit(int u, uint4& x, u32 parent, u32 own_edge) {
        if (u == 1) { x.z = parent; x.w = own_edge; }
        else if (u == 2) x.y &= ~META_EXPANDED;
    }
    __device__ static void load_links(const uint4* p, u32& parent, u32& own_edge) { uint4 b = p[1]; parent = b.z; own_edge = b.w; }
    __device__ static void load_boards(const uint4* p, Bits<1>& b0, Bits<1>& b1) {
        uint4 a = p[0];
        b0 = Bits<1>((u64)a.x | ((u64)a.y << 32));
        b1 = Bits<1>((u64)a.z | ((u64)a.w << 32));
    }
};
template <> struct HL<2> {
    static constexpr int HDR = 5;
    __device__ static Bits<2> bits(uint4 a) { return Bits<2>((u64)a.x | ((u64)a.y << 32), (u64)a.z | ((u64)a.w << 32)); }
    __device__ static uint4 unit(const Bits<2>& b) { return make_uint4((u32)b.w0, (u32)(b.w0 >> 32), (u32)b.w1, (u32)(b.w1 >> 32)); }
    __device__ static void load(const uint4* p, Hdr<2>& h) {
        h.b0 = bits(p[0]); h.b1 = bits(p[1]); h.legal = bits(p[2]);
        uint4 d = p[3], e = p[4];
        h.parent = d.x; h.own_edge = d.y; h.net_value = __uint_as_float(d.z); h.meta = d.w; h.aux = e.x;
    }
    __device__ static void store_unit(uint4* p, int i, const Hdr<2>& h) {
        if (i == 0) p[0] = unit(h.b0);
        else if (i == 1) p[1] = unit(h.b1);
        else if (i == 2) p[2] = unit(h.legal);
        else if (i == 3) p[3] = make_uint4(h.parent, h.own_edge, __float_as_uint(h.net_value), h.meta);
        else p[4] = make_uint4(h.aux, 0u, 0u, 0u);
    }
    __device__ static u32* meta_ptr(uint4* p) { return reinterpret_cast<u32*>(p + 3) + 3; }
    __device__ static float* value_ptr(uint4* p) { return reinterpret_cast<float*>(p + 3) + 2; }
    __device__ static void relink_unit(int u, uint4& x, u32 parent, u32 own_edge) {
        if (u == 3) { x.x = parent; x.y = own_edge; x.w &= ~META_EXPANDED; }
    }
    __device__ static void load_links(const uint4* p, u32& parent, u32& own_edge) { uint4 d = p[3]; parent = d.x; own_edge = d.y; }
    __device__ static void load_boards(const uint4* p, Bits<2>& b0, Bits<2>& b1) { b0 = bits(p[0]); b1 = bits(p[1]); }
};

template <class G>
__device__ __forceinline__ void pos_to_hdr(const typename G::P& p, u32 parent, u32 own_edge, Hdr<G::W>& h) {
    h.b0 = p.b[0]; h.b1 = p.b[1]; h.legal = p.legal;
    h.parent = parent; h.own_edge = own_edge; h.net_value = 0.0f;
    u32 n = p.terminal ? 0u : (u32)p.n_legal();          // edges exist only below non-terminal nodes
    h.meta = n | ((u32)p.player << 8) | ((u32)p.terminal << 9) | ((u32)p.winner << 10) |
             ((u32)p.pass_legal << 14) | ((u32)p.action << 16);
    h.aux = p.depth;
}
template <class G>
__device__ __forceinline__ void hdr_to_pos(const Hdr<G::W>& h, typename G::P& p) {
    p.b[0] = h.b0; p.b[1] = h.b1; p.legal = h.legal;
    p.player = META_PLAYER(h.meta); p.terminal = META_TERMINAL(h.meta); p.winner = META_WINNER(h.meta);
    p.pass_legal = META_PASS_LEGAL(h.meta); p.action = META_ACTION(h.meta); p.depth = (unsigned short)h.aux;
}

// shared-memory scratch of one warp
constexpr int DESCENT_MAX = 32;        // edges of a descent recorded for the parallel backup (deeper ones walk parent links)
struct WarpScratch {
    float pol[96];      // dense per-action vector (policy / pdf)
    float aux[96];      // per-slot vector (noise, cdf)
    u32 path[DESCENT_MAX]; // own edges of the nodes on the last descent, root first: path[0] = the tree's dummy edge (unit 0)
};

// ---- the warp that owns a tree -----------------------------------------------------------------
template <class G, bool MATCH = false>
struct TreeWarp {
    static constexpr int W = G::W;
    static constexpr int HDR = HL<W>::HDR;
    static constexpr int NCH = (G::ACTIONS + 31) / 32;
    typedef Hdr<W> H;
    typedef typename G::P P;

    // registers of the owning warp: the hot part of TreeState; counters are accumulated
    // locally (32-bit) and added to the tree's record once per launch
    struct Hot {
        unsigned long long game_id;
        u32 n_units, slab, high_water;
        int traversals, move_count, status, n_queued;
        long long game_index;
    };
    struct Acc { u32 sims, evals, moves, games, depth_sum, legal_sum, nodes_visited, leaves_terminal, leaves_gray, leaves_empty, leaves_duplicate; };

    const EngineParams& p;
    const int tree, lane;
    Hot st;
    Acc acc;
    Rng rng;
    uint4* slab;            // current slab
    WarpScratch& sm;
    AgentCfg agent;         // match play: this side's evaluator / symmetrizer / init-Q (unused in self-play)
    int sel_edges;          // own edges recorded in sm.path by the last select_leaf (0: the descent was deeper than DESCENT_MAX)
    int game_step;          // game_index stride: slots (self-play) or pairs (match play)

    // per-tree options: the engine's in self-play, the side's in match play
    __device__ __forceinline__ int cfg_evaluator() const { if constexpr (MATCH) return agent.evaluator; else return p.evaluator; }
    __device__ __forceinline__ int cfg_use_sym() const { if constexpr (MATCH) return agent.use_sym; else return p.use_sym; }
    __device__ __forceinline__ int cfg_init_q() const { if constexpr (MATCH) return agent.init_q; else return p.init_q; }
    __device__ __forceinline__ unsigned long long cfg_salt() const { if constexpr (MATCH) return agent.hash_salt; else return 0ULL; }

    __device__ TreeWarp(const EngineParams& p_, int tree_, int lane_, WarpScratch& sm_, const AgentCfg* agent_ = nullptr, int game_step_ = 0)
        : p(p_), tree(tree_), lane(lane_), sm(sm_) {
        if constexpr (MATCH) { agent = *agent_; game_step = game_step_; } else { game_step = p_.n_slots; }
        const TreeState& g = p.trees[tree];
        st.game_id = g.game_id; st.n_units = g.n_units; st.slab = g.slab; st.high_water = g.high_water;
        st.traversals = g.traversals; st.move_count = g.move_count; st.status = g.status; st.n_queued = g.n_queued;
        st.game_index = g.game_index;
        acc = Acc{ 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
        rng.seed = p.seed; rng.game = st.game_id; rng.ctr = g.rng_ctr;
        slab = slab_ptr(st.slab);
    }
    __device__ uint4* slab_ptr(u32 which) const { return p.pool + ((size_t)tree * 2 + which) * p.cap_units; }
    __device__ void save() {
        if (st.n_units > st.high_water) st.high_water = st.n_units;
        if (lane == 0) {
            TreeState& g = p.trees[tree];
            g.game_id = st.game_id; g.rng_ctr = rng.ctr; g.n_units = st.n_units; g.slab = st.slab;
            g.high_water = st.high_water; g.traversals = st.traversals; g.move_count = st.move_count;
            g.status = st.status; g.n_queued = st.n_queued; g.game_index = st.game_index;
            g.sims += acc.sims; g.evals += acc.evals; g.moves += acc.moves; g.games += acc.games;
            g.depth_sum += acc.depth_sum; g.legal_sum += acc.legal_sum; g.nodes_visited += acc.nodes_visited;
            g.leaves_terminal += acc.leaves_terminal; g.leaves_gray += acc.leaves_gray; g.leaves_empty += acc.leaves_empty;
            g.leaves_duplicate += acc.leaves_duplicate;
        }
    }
    __device__ size_t rec_index() const { return (size_t)st.game_index * p.max_moves + st.move_count; }

    // ---- history of boards above a node: tree ancestors, then the game's earlier moves ----
    struct TreeHist {
        const TreeWarp* t;
        u32 start;          // first unit whose board is compared (walks parent links to the root)
        __device__ bool seen(const Bits<W>& a0, const Bits<W>& a1) const {
            u32 cur = start;
            for (;;) {
                Bits<W> b0, b1;
                HL<W>::load_boards(t->slab + cur, b0, b1);
                if (b0 == a0 && b1 == a1) return true;
                if (cur == ROOT_UNIT) break;
                u32 par, own;
                HL<W>::load_links(t->slab + cur, par, own);
                cur = par;
            }
            const unsigned long long* rb = t->p.rec_board + (size_t)t->st.game_index * t->p.max_moves * 2 * W;
            for (int m = t->st.move_count - 1; m >= 0; --m) {
                bool same = true;
                for (int w = 0; w < W; ++w)
                    same = same && rb[(size_t)m * 2 * W + w] == a0.word(w) && rb[(size_t)m * 2 * W + W + w] == a1.word(w);
                if (same) return true;
            }
            return false;
        }
        template <class F> __device__ void for_each(F&& f) const {
            u32 cur = start;
            for (;;) {
                Bits<W> b0, b1;
                HL<W>::load_boards(t->slab + cur, b0, b1);
                f(b0, b1);
                if (cur == ROOT_UNIT) break;
                u32 par, own;
                HL<W>::load_links(t->slab + cur, par, own);
                cur = par;
            }
            const unsigned long long* rb = t->p.rec_board + (size_t)t->st.game_index * t->p.max_moves * 2 * W;
            for (int mv = t->st.move_count - 1; mv >= 0; --mv) {
                Bits<W> b0, b1;
                for (int w = 0; w < W; ++w) { b0.set_word(w, rb[(size_t)mv * 2 * W + w]); b1.set_word(w, rb[(size_t)mv * 2 * W + W + w]); }
                f(b0, b1);
            }
        }
    };

    // boards of the position `t` plies above `unit` (0 = itself); false when the game is younger
    __device__ bool history_board(u32 unit, int t, Bits<W>& b0, Bits<W>& b1) const {
        u32 cur = unit;
        while (t > 0 && cur != ROOT_UNIT) {
            u32 par, own;
            HL<W>::load_links(slab + cur, par, own);
            cur = par; --t;
        }
        if (t == 0) { HL<W>::load_boards(slab + cur, b0, b1); return true; }
        int m = st.move_count - t;
        if (m < 0) return false;
        const unsigned long long* rb = p.rec_board + ((size_t)st.game_index * p.max_moves + m) * 2 * W;
        for (int w = 0; w < W; ++w) { b0.set_word(w, rb[w]); b1.set_word(w, rb[W + w]); }
        return true;
    }

    // ---- GameNode::getNextNodeImpl for the child of `par` (unit par_unit) ----
    __device__ void make_child_pos(const P& par, u32 par_unit, int action, P& child) {
        if constexpr (G::KIND == GAME_GO7 || G::KIND == GAME_GO9) {
            G::template next_board<NoHistory>(par, action, child);
            if (!child.terminal) {
                // Legal placements of the new position (checkLegalPlacement, games/GoNode.cpp:178-228) for all points at once
                // (Go::legal_from_groups).  The group scan is spread over the warp: every lane floods the groups of its own
                // cells and the liberty sets are OR-ed across the lanes; the rest is warp-uniform.  Superko compares against
                // the new board itself, `par` and everything above it.
                const typename G::Masks m = G::masks();
                const Bits<W> own = child.b[child.player], opp = child.b[1 - child.player], empty = m.all & ~(own | opp);
                Bits<W> own_multi, own_atari, opp_multi, opp_atari;
                for (int base = 0; base < G::CELLS; base += 32) {
                    const int c = base + lane;
                    if (c < G::CELLS) {
                        if (own.test(c)) G::group_liberties(Bits<W>::bit(c), own, empty, m, own_multi, own_atari);
                        else if (opp.test(c)) G::group_liberties(Bits<W>::bit(c), opp, empty, m, opp_multi, opp_atari);
                    }
                }
                own_multi = warp_or(own_multi);
                opp_atari = warp_or(opp_atari);
                const TreeHist th = { this, par_unit };
                const HistPlus<TreeHist, W> hist = { th, child.b[0], child.b[1] };
                child.legal = G::legal_from_groups(own, opp, child.player, m, hist, own_multi, opp_atari);
            }
        } else if constexpr (G::KIND == GAME_OTHELLO) {
            G::next_warp(par, action, lane, child);          // called by the whole warp with uniform arguments
        } else {
            G::next(par, action, NoHistory(), child);
        }
    }
    // OR of a bit set over the lanes of the warp
    __device__ static Bits<W> warp_or(const Bits<W>& x) {
        Bits<W> r;
        for (int w = 0; w < W; ++w) {
            const u64 v = x.word(w);
            const u32 lo = __reduce_or_sync(FULL, (u32)v), hi = __reduce_or_sync(FULL, (u32)(v >> 32));
            r.set_word(w, (u64)lo | ((u64)hi << 32));
        }
        return r;
    }
    // 32 cells [base, base+32) of a bit set, from a warp ballot
    __device__ static Bits<W> from_ballot(u32 bal, int base) {
        Bits<W> r;
        if (base < 64) r.set_word(0, (u64)bal << base);
        else if constexpr (W == 2) r.set_word(1, (u64)bal << (base - 64));
        return r;
    }

    // ---- writes a node record at `unit`; all lanes hold `child` ----
    __device__ bool write_node(uint4* dst_slab, u32 unit, const P& child, u32 parent, u32 own_edge, H& h) {
        pos_to_hdr<G>(child, parent, own_edge, h);
        int n = META_NLEGAL(h.meta);
        if (lane < HDR) HL<W>::store_unit(dst_slab + unit, lane, h);
        for (int base = 0; base < n; base += 32) {
            int k = base + lane;
            if (k < n) {
                u32 a = (u32)legal_action<G>(child, k);
                dst_slab[unit + HDR + k] = make_uint4(0u, 0u, 0u, a << 24);
            }
        }
        return true;
    }

    // ---- the game starts from its opening line, as if the caller had advanced a fresh tree through it: the line's
    //      positions become the game's recorded history (later network inputs, samples, superko), the position it ends in
    //      becomes the root.  Returns the line's length. ----
    __device__ int open_line(long long n_lines, P& pos) {
        const unsigned long long t = MATCH ? st.game_id / 2 : st.game_id;     // match play: both colour assignments of a line
        const int line = (int)(t % (unsigned long long)n_lines);
        const int a0 = (int)p.iter->open_off[line];
        const int len = (int)p.iter->open_off[line + 1] - a0;
        const PosRec* r = p.iter->open_rec + a0 + line;
        unsigned long long* rb = p.rec_board + (size_t)st.game_index * p.max_moves * 2 * W;
        unsigned char* rp = p.rec_player + (size_t)st.game_index * p.max_moves;
        for (int k = lane; k < len; k += 32) {
            for (int w = 0; w < W; ++w) { rb[k * 2 * W + w] = r[k].b[w]; rb[k * 2 * W + W + w] = r[k].b[2 + w]; }
            rp[k] = r[k].player;
        }
        rec_to_pos<G>(r[len], pos);
        return len;
    }

    __device__ void init_game() {
        st.game_id = p.iter->first_game + (unsigned long long)st.game_index * p.iter->game_stride;
        rng.game = st.game_id; rng.ctr = 0;
        st.slab = 0; slab = slab_ptr(0);
        st.traversals = 0; st.move_count = 0; st.n_queued = 0;
        const long long n_lines = p.iter->n_lines;
        H h;
        if (lane == 0) slab[0] = make_uint4(0u, 0u, 0u, 0u);
        if (n_lines > 0) {
            P pos;
            st.move_count = open_line(n_lines, pos);
            write_node(slab, ROOT_UNIT, pos, 0u, 0u, h);
        } else {
            P start;
            G::start(start);
            write_node(slab, ROOT_UNIT, start, 0u, 0u, h);
        }
        if (lane == 0) p.rec_open[st.game_index] = st.move_count;
        st.n_units = ROOT_UNIT + HDR + META_NLEGAL(h.meta);
        __syncwarp();
    }

    // ---- UCTTree::backup (uct/UCTTree.hpp:261-273) by walking parent links ----
    // With the descent's own edges at hand (n_path of them, root first) every level is updated by its own lane: the W's
    // of one backup are distinct words, and each update is the reference's `W += 1 + estimate * sign(player)`.
    __device__ void backup_path(const u32* path, int n_path, int leaf_player, float value) {
        const float est = -value * (leaf_player == 0 ? 1.0f : -1.0f);
        if (lane < n_path) {
            const int up = n_path - 1 - lane;                       // plies above the leaf: players alternate
            const float term = 1.0f + est * (((leaf_player ^ up) & 1) == 0 ? 1.0f : -1.0f);
            float* w = reinterpret_cast<float*>(slab + path[lane]) + 1;
            *w = *w + term;
        }
        __syncwarp();
    }
    __device__ void backup(u32 leaf, int leaf_player, float value) {
        float est = -value * (leaf_player == 0 ? 1.0f : -1.0f);
        u32 cur = leaf;
        int player = leaf_player;
        for (;;) {
            u32 par, own;
            HL<W>::load_links(slab + cur, par, own);
            float term = 1.0f + est * (player == 0 ? 1.0f : -1.0f);
            if (lane == 0) {
                float* w = reinterpret_cast<float*>(slab + own) + 1;
                *w = *w + term;
            }
            if (cur == ROOT_UNIT) break;
            cur = par; player ^= 1;
        }
        __syncwarp();
    }

    // ---- Dirichlet mix at the decision node (uct/UCTNode.hpp:330-346) ----
    __device__ void root_noise(int n) {
        float sum = 0.0f;
        for (int k = 0; k < n; ++k) {                    // sequential stream: every lane draws the same values
            float g = rng_gamma(rng, p.dir_alpha);
            if (lane == 0) sm.aux[k] = g;
            sum += g;
        }
        float norm = 1.0f / sum;
        __syncwarp();
        for (int base = 0; base < n; base += 32) {
            int k = base + lane;
            if (k < n) {
                float noise = sm.aux[k] * norm;
                float prior = __uint_as_float(slab[ROOT_UNIT + HDR + k].x);
                float mixed = (float)((1.0 - (double)p.dir_eps) * (double)prior + (double)(p.dir_eps * noise));
                p.root_p[(size_t)tree * G::ACTIONS + k] = mixed;
            }
        }
        __syncwarp();
    }

    // ---- UCTNode::expand (uct/UCTNode.hpp:314-348): gray -> active ----
    __device__ void expand(u32 unit, u32& meta) {
        meta |= META_EXPANDED;
        if (lane == 0) *HL<W>::meta_ptr(slab + unit) = meta;
        if (unit == ROOT_UNIT && p.add_noise) root_noise(META_NLEGAL(meta));
        __syncwarp();
    }

    // ---- one descent: UCTTree::selectLeaf (uct/UCTTree.hpp:225-249) ----
    // Virtual loss (N += 1, W -= 1) is written on the edge INTO a node at the moment
    // the edge is chosen; the pre-loss N of that edge is what the child's sqrt(N()) uses.
    __device__ u32 select_leaf(H& leaf_hdr) {
        u32 cur = ROOT_UNIT;
        uint4 d = slab[0];
        float n_own = __uint_as_float(d.z);
        // InitQ::DROP_PARENT (uct/UCTNode.hpp:152-163,196-206): W, N of the current node before this descent's
        // virtual loss, and the Q of its parent after it (the answer of an unvisited node; never needed in
        // practice, a node is visited before it is expanded)
        const bool drop = cfg_init_q() == SPRL_INITQ_DROP_PARENT;
        float w_own = __uint_as_float(d.y), q_par = 0.0f;
        if (lane == 0) slab[0] = make_uint4(d.x, __float_as_uint(__uint_as_float(d.y) - 1.0f), __float_as_uint(n_own + 1.0f), d.w);
        int depth = 0;
        bool have = false;
        H h;
        if (lane == 0) sm.path[0] = 0u;                 // the root's own edge is the tree's dummy edge
        for (;;) {
            if (!have) HL<W>::load(slab + cur, h);
            have = false;
            if (META_TERMINAL(h.meta) || !(h.meta & META_EXPANDED)) break;
            const int n = META_NLEGAL(h.meta);
            acc.nodes_visited += 1; acc.legal_sum += n;
            // UCTNode::bestAction (uct/UCTNode.hpp:221-251)
            const float sq = sqrtf(n_own);
            float q_own = 0.0f;
            if (drop) q_own = (n_own == 0.0f) ? q_par : w_own / n_own;
            uint4 e[NCH];
            float val[NCH];
            float best = -__int_as_float(0x7f800000);
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                int k = ch * 32 + lane;
                val[ch] = -__int_as_float(0x7f800000);
                if (k < n) {
                    e[ch] = slab[cur + HDR + k];
                    float prior = (cur == ROOT_UNIT && p.add_noise) ? p.root_p[(size_t)tree * G::ACTIONS + k] : __uint_as_float(e[ch].x);
                    float w = __uint_as_float(e[ch].y), nv = __uint_as_float(e[ch].z);
                    float q = w / (1.0f + nv);
                    if (drop) q = (nv == 0.0f) ? q_own : w / nv;
                    float u = prior * sq / (1.0f + nv);
                    val[ch] = q + p.u_weight * u;
                }
                best = fmaxf(best, val[ch]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(FULL, best, o));
            u32 bal[NCH];
            int cnt = 0;
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                bal[ch] = __ballot_sync(FULL, (ch * 32 + lane < n) && val[ch] == best);
                cnt += __popc(bal[ch]);
            }
            int r = rng_uniform_int(rng, 0, cnt - 1);       // tie-break, uct/UCTNode.hpp:250
            int ksel = 0;
            bool found = false;
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                int c = __popc(bal[ch]);
                if (!found && r < c) { ksel = ch * 32 + (r == 0 ? __ffs((int)bal[ch]) - 1 : nth_set_bit32(bal[ch], r)); found = true; }
                if (!found) r -= c;
            }
            uint4 es = e[0];
#pragma unroll
            for (int ch = 1; ch < NCH; ++ch) if ((ksel >> 5) == ch) es = e[ch];
            const int src_lane = ksel & 31;
            u32 ew = __shfl_sync(FULL, es.w, src_lane);
            float child_n = __uint_as_float(__shfl_sync(FULL, es.z, src_lane));
            u32 child = EDGE_CHILD(ew);
            const u32 edge_unit = cur + HDR + ksel;
            float w_sel = __uint_as_float(es.y);
            if (child == 0) {
                // UCTNode::getAddChild (uct/UCTNode.hpp:258-284) + GameNode::getAddChild
                P par, cp;
                hdr_to_pos<G>(h, par);
                make_child_pos(par, cur, (int)EDGE_ACTION(ew), cp);
                u32 need = HDR + (cp.terminal ? 0u : (u32)cp.n_legal());
                if (st.n_units + need + SLAB_SLACK > p.cap_units) { st.status = ST_ERR_CAPACITY; leaf_hdr = h; return cur; }
                child = st.n_units;
                st.n_units += need;
                H ch;
                write_node(slab, child, cp, cur, edge_unit, ch);
                ew |= child;
                w_sel = (cfg_init_q() == SPRL_INITQ_PARENT && (h.meta & META_EVALUATED)) ? h.net_value : 0.0f;
                h = ch; have = true;
            }
            if (drop) { q_par = (w_own - 1.0f) / (n_own + 1.0f); w_own = __shfl_sync(FULL, w_sel, src_lane); }
            if (lane == src_lane)
                slab[edge_unit] = make_uint4(es.x, __float_as_uint(w_sel - 1.0f), __float_as_uint(child_n + 1.0f), ew);
            n_own = child_n;
            cur = child;
            ++depth;
            if (lane == 0 && depth < DESCENT_MAX) sm.path[depth] = edge_unit;
            __syncwarp();
        }
        acc.depth_sum += depth;
        sel_edges = depth < DESCENT_MAX ? depth + 1 : 0;
        leaf_hdr = h;
        return cur;
    }

    // ---- UCTTree::searchAndGetLeaves (uct/UCTTree.hpp:76-114) + the symmetry draws of :141-149 ----
    __device__ void search_batch() {
        int trav = 0, nq = 0;
        u32 my_leaf = 0;                                // lane q < 32 remembers queue entry q
        while (trav < p.max_batch) {
            ++trav;
            H h;
            u32 leaf = select_leaf(h);
            if (st.status != ST_PLAYING) return;
            int player = META_PLAYER(h.meta);
            if (META_TERMINAL(h.meta)) {
                u32 wn = META_WINNER(h.meta);
                float value = (wn == WINNER_NONE) ? 0.0f : ((int)wn - 1 == player ? 1.0f : -1.0f);
                if (sel_edges) backup_path(sm.path, sel_edges, player, value); else backup(leaf, player, value);
                acc.leaves_terminal += 1;
                continue;
            } else if (h.meta & META_EVALUATED) {
                expand(leaf, h.meta);
                if (sel_edges) backup_path(sm.path, sel_edges, player, h.net_value); else backup(leaf, player, h.net_value);
                acc.leaves_gray += 1;
                continue;
            } else {
                const size_t qs = (size_t)tree * p.max_queue + nq;
                if (lane == 0) { p.q_leaf[qs] = leaf; p.q_plen[qs] = (unsigned char)sel_edges; }
                if (lane < sel_edges) p.q_path[qs * DESCENT_MAX + lane] = sm.path[lane];      // for the backup in the next launch
                if (lane == nq) my_leaf = leaf;
                ++nq;
                acc.leaves_empty += 1;
            }
            if (nq >= p.max_queue) break;
        }
        st.traversals += trav;
        acc.sims += trav;
        st.n_queued = nq;
        __syncwarp();
        // Quirk Q4 (uct/UCTTree.hpp:166-182): a node can be queued several times in one batch; every copy gets a symmetry
        // draw and is backed up, but only the FIRST evaluation is kept -- so only the first copy gets an evaluator row.
        // (Entries beyond the 32nd of a very wide queue are not compared: each keeps its own row.)
        const int n32 = min(nq, 32);
        bool dup = false;
        for (int k = 0; k + 1 < n32; ++k) {
            const u32 v = __shfl_sync(FULL, my_leaf, k);
            dup = dup || (lane > k && lane < n32 && my_leaf == v);
        }
        const u32 first_mask = __ballot_sync(FULL, lane < n32 && !dup);
        const int n_rows = __popc(first_mask) + (nq - n32);
        acc.leaves_duplicate += (u32)(nq - n_rows);
        u32 row0 = 0;                                   // rows of the evaluator batch for this tree's leaves
        if (cfg_evaluator() == SPRL_EVAL_EXTERNAL && nq > 0) {
            const int side = MATCH ? agent.pad : 0;
            if (lane == 0) row0 = atomicAdd(&p.q_count[side], (u32)n_rows) + (side ? p.iter->q_half : 0u);
            row0 = __shfl_sync(FULL, row0, 0);
            if (lane == 0) p.q_base[tree] = row0;
        }
        for (int q = 0; q < nq; ++q) {
            int s = cfg_use_sym() ? rng_uniform_int(rng, 0, G::NSYM - 1) : 0;
            const bool first = q >= 32 || ((first_mask >> q) & 1u);
            const u32 off = q >= 32 ? (u32)(__popc(first_mask) + q - 32) : (u32)__popc(first_mask & ((1u << q) - 1u));
            if (lane == 0) { p.q_sym[(size_t)tree * p.max_queue + q] = (unsigned char)s; p.q_rowoff[(size_t)tree * p.max_queue + q] = (unsigned char)off; }
            if (first && cfg_evaluator() == SPRL_EVAL_EXTERNAL) encode_leaf(p.q_leaf[(size_t)tree * p.max_queue + q], s, (size_t)row0 + off);
        }
        acc.evals += nq;
        __syncwarp();
    }

    // ---- network input planes of a leaf under symmetry s (networks/GridNetwork.hpp:72-97) ----
    __device__ void encode_leaf(u32 unit, int s, size_t slot) {
        constexpr int PLANES = 2 * G::HISTORY + 1;
        float* out = p.nn_in + slot * PLANES * G::CELLS;
        u32 meta = *HL<W>::meta_ptr(slab + unit);
        int player = META_PLAYER(meta);
        int inv = sym_inverse<G>(s);
        for (int t = 0; t < G::HISTORY; ++t) {
            Bits<W> b0, b1;
            bool valid = history_board(unit, t, b0, b1);
            const Bits<W>& own = player == 0 ? b0 : b1;
            const Bits<W>& opp = player == 0 ? b1 : b0;
            for (int to = lane; to < G::CELLS; to += 32) {
                int from = sym_cell<G>(inv, to);
                out[(2 * t) * G::CELLS + to] = (valid && own.test(from)) ? 1.0f : 0.0f;
                out[(2 * t + 1) * G::CELLS + to] = (valid && opp.test(from)) ? 1.0f : 0.0f;
            }
        }
        for (int to = lane; to < G::CELLS; to += 32) out[(PLANES - 1) * G::CELLS + to] = player == 0 ? 1.0f : 0.0f;
    }

    // symmetrised bitboard: bit f_s(i) of the result = bit i of x
    __device__ Bits<W> sym_bits(const Bits<W>& x, int s) {
        int inv = sym_inverse<G>(s);
        Bits<W> r;
        for (int base = 0; base < G::CELLS; base += 32) {
            int to = base + lane;
            bool bit = to < G::CELLS && x.test(sym_cell<G>(inv, to));
            u32 bal = __ballot_sync(FULL, bit);
            r = r | from_ballot(bal, base);
        }
        return r;
    }

    // hash of the symmetrised input state (HashNet, shared definition with the oracle)
    __device__ unsigned long long state_hash(u32 unit, int player, int s) {
        unsigned long long h = hashnet_seed(player);
        for (int t = 0; t < G::HISTORY; ++t) {
            Bits<W> b0, b1;
            if (!history_board(unit, t, b0, b1)) break;
            Bits<W> own = sym_bits(player == 0 ? b0 : b1, s), opp = sym_bits(player == 0 ? b1 : b0, s);
            h = hash_mix(h ^ own.word(0));
            h = hash_mix(h ^ (W == 2 ? own.word(W - 1) : 0ULL));
            h = hash_mix(h ^ opp.word(0));
            h = hash_mix(h ^ (W == 2 ? opp.word(W - 1) : 0ULL));
        }
        return h;
    }

    // ---- INetwork::evaluate for one leaf + inverse symmetry + UCTNode::addNetworkOutput ----
    // Policy entries live in the SYMMETRISED frame but are masked with the leaf's
    // un-symmetrised mask (uct/UCTTree.hpp:136-149, networks/GridNetwork.hpp:117-125:
    // reference quirk Q3), then mapped back with the inverse symmetry.
    __device__ void evaluate_leaf(u32 unit, H& h, int s, size_t slot) {
        const int n = META_NLEGAL(h.meta);
        const int player = META_PLAYER(h.meta);
        P pos;
        hdr_to_pos<G>(h, pos);
        // the legal mask the evaluator applies to its (symmetrised-frame) policy: the reference hands it the
        // UN-symmetrised one (quirk Q3); with fix_symmetry_mask it is symmetrised like the state
        P mpos = pos;
        if (p.fix_symmetry_mask && cfg_use_sym()) mpos.legal = sym_bits(pos.legal, s);
        float value = 0.0f;
        for (int i = lane; i < G::ACTIONS; i += 32) sm.pol[i] = 0.0f;
        __syncwarp();
        const int ev = cfg_evaluator();
        if (ev == SPRL_EVAL_UNIFORM || ev == SPRL_EVAL_OTHELLO_HEURISTIC) {   // networks/RandomNetwork.hpp:21-49
            float uniform = 1.0f / (float)n;
            for (int base = 0; base < n; base += 32) {
                int k = base + lane;
                if (k < n) sm.pol[legal_action<G>(mpos, k)] = uniform;
            }
            __syncwarp();
            if constexpr (G::KIND == GAME_OTHELLO) {
                if (ev == SPRL_EVAL_OTHELLO_HEURISTIC) {
                    // networks/OthelloHeuristic.cpp:18-50: (own legal actions, the pass slot included, minus the
                    // opponent's placements) / empty squares; all three counts are symmetry-invariant
                    const u64 own = player == 0 ? h.b0.w0 : h.b1.w0, opp = player == 0 ? h.b1.w0 : h.b0.w0;
                    const int num_opp = __popcll(Othello::mobility(opp, own));
                    const int num_empty = 64 - __popcll(own | opp);
                    value = (float)(n - num_opp) / (float)num_empty;
                }
            }
        } else {
            unsigned long long hh = 0;
            if (ev == SPRL_EVAL_HASHNET) { hh = hashnet_salt(state_hash(unit, player, s), cfg_salt()); value = hashnet_value(hh); }
            else value = p.nn_value[slot];
            // Each lane holds the raw prior of its k-th legal action; GameActionDist::sum adds them in ascending
            // index order = ascending k, done with one shuffle per element.  Up to 32 legal actions (the usual
            // case) the values stay in registers until they are normalised.
            float sum = 0.0f, v = 0.0f;
            int i = 0;
            for (int base = 0; base < n; base += 32) {
                const int k = base + lane;
                v = 0.0f;
                if (k < n) {
                    i = legal_action<G>(mpos, k);           // mask index == policy index (symmetrised frame)
                    v = (ev == SPRL_EVAL_HASHNET) ? hashnet_prior_raw(hh, i)
                                                  : det_expf(p.nn_logits[slot * G::ACTIONS + i]);
                    if (n > 32) sm.pol[i] = v;
                }
                const int cnt = min(32, n - base);
                for (int j = 0; j < cnt; ++j) sum += __shfl_sync(FULL, v, j);
            }
            const float uniform = 1.0f / (float)n;
            const float inv = 1.0f / sum;                    // operator/(dist, float) = multiply by the reciprocal
            if (n <= 32) {
                if (lane < n) sm.pol[i] = (sum == 0.0f) ? uniform : v * inv;
            } else {
                for (int base = 0; base < n; base += 32) {
                    const int k = base + lane;
                    if (k < n) { i = legal_action<G>(mpos, k); sm.pol[i] = (sum == 0.0f) ? uniform : sm.pol[i] * inv; }
                }
            }
            __syncwarp();
        }
        // inverse symmetry: prior of action a = policy[f_s(a)]
        for (int base = 0; base < n; base += 32) {
            int k = base + lane;
            if (k < n) {
                int a = legal_action<G>(pos, k);
                float prior = sm.pol[cfg_use_sym() ? sym_action<G>(s, a) : a];
                reinterpret_cast<float*>(slab + unit + HDR + k)[0] = prior;
            }
        }
        h.net_value = value;
        h.meta |= META_EVALUATED;
        if (lane == 0) { *HL<W>::value_ptr(slab + unit) = value; *HL<W>::meta_ptr(slab + unit) = h.meta; }
        __syncwarp();
    }

    // ---- UCTTree::evaluateAndBackpropLeaves (uct/UCTTree.hpp:154-183) ----
    __device__ void apply_leaves() {
        const size_t row0 = cfg_evaluator() == SPRL_EVAL_EXTERNAL ? (size_t)p.q_base[tree] : 0;
        for (int q = 0; q < st.n_queued; ++q) {
            size_t slot = (size_t)tree * p.max_queue + q;
            u32 leaf = p.q_leaf[slot];
            int s = p.q_sym[slot];
            H h;
            HL<W>::load(slab + leaf, h);
            if (!(h.meta & META_EVALUATED)) evaluate_leaf(leaf, h, s, row0 + p.q_rowoff[slot]);
            if (!(h.meta & META_EXPANDED)) expand(leaf, h.meta);
            const int n_path = p.q_plen[slot];
            if (n_path) backup_path(p.q_path + slot * DESCENT_MAX, n_path, META_PLAYER(h.meta), h.net_value);
            else backup(leaf, META_PLAYER(h.meta), h.net_value);
        }
        st.n_queued = 0;
    }

    // ---- copies the subtree below src unit `c` into the other slab (UCTTree::advanceDecision,
    //      pruneChildrenExcept + clearSubtree, uct/UCTTree.hpp:197-210,283-298) ----
    // Breadth-first, so parents precede children and siblings end up adjacent.  Every copied edge
    // restarts with W = N = 0 and every node un-expanded; cached evaluations (netP, net_value,
    // evaluated bit) are kept.  The frontier is a FIFO of child links (parent record << 8 | edge
    // slot) in HBM; each step takes up to 32 links, sizes the 32 child records with one warp scan,
    // copies all their units with the whole warp (flat unit index -> record by a shuffle binary
    // search, so the loads of a step are independent) and appends the links found in them.
    __device__ bool compact_into(uint4* dst, u32 c, float own_w, float own_n, u32& out_units) {
        if (lane == 0) dst[0] = make_uint4(0u, __float_as_uint(own_w), __float_as_uint(own_n), 0u);
        u32* q = p.cq + (size_t)tree * p.cq_cap;
        u32 head = 0, tail = 0, alloc = ROOT_UNIT;
        bool root_step = true;
        for (;;) {
            const int n = root_step ? 1 : (int)min(32u, tail - head);
            // ---- one record per lane: where it comes from, how big it is
            u32 src = 0, size = 0, parent = 0, own_edge = 0, ew = 0;
            if (lane < n) {
                if (root_step) src = c;
                else {
                    const u32 link = q[head + lane];
                    parent = link >> 8;
                    own_edge = parent + HDR + (link & 0xffu);
                    ew = dst[own_edge].w;
                    src = EDGE_CHILD(ew);
                }
                size = HDR + META_NLEGAL(*HL<W>::meta_ptr(slab + src));
            }
            u32 incl = size;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                u32 v = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += v;
            }
            const u32 total = __shfl_sync(FULL, incl, 31);
            if (alloc + total + SLAB_SLACK > p.cap_units) return false;
            const u32 nu = alloc + incl - size;                          // new home of this lane's record
            if (lane < n && !root_step) reinterpret_cast<u32*>(dst + own_edge)[3] = (ew & 0xff000000u) | nu;
            // ---- copy: flat unit x of the step belongs to the first record r with incl[r] > x
#pragma unroll 2
            for (u32 x0 = 0; x0 < total; x0 += 32) {                     // every lane runs every trip (shuffles)
                const u32 x = x0 + lane;
                int lo = 0, hi = 31;
#pragma unroll
                for (int it = 0; it < 5; ++it) {
                    const int mid = (lo + hi) >> 1;
                    const u32 v = __shfl_sync(FULL, incl, mid);
                    if (v > x) hi = mid; else lo = mid + 1;
                }
                const u32 r_incl = __shfl_sync(FULL, incl, lo), r_size = __shfl_sync(FULL, size, lo);
                const u32 r_src = __shfl_sync(FULL, src, lo), r_nu = __shfl_sync(FULL, nu, lo);
                const u32 r_parent = __shfl_sync(FULL, parent, lo), r_edge = __shfl_sync(FULL, own_edge, lo);
                if (x < total) {
                    const u32 u = x - (r_incl - r_size);
                    uint4 v = slab[r_src + u];
                    if (u < (u32)HDR) HL<W>::relink_unit((int)u, v, r_parent, r_edge);
                    else { v.y = 0u; v.z = 0u; }
                    dst[r_nu + u] = v;
                }
            }
            __syncwarp();
            // ---- links of the copied records, in record order then edge order
            u32 links = 0;
            if (lane < n) {
                const int cn = (int)size - HDR;
                for (int j = 0; j < cn; ++j) links += EDGE_CHILD(slab[src + HDR + j].w) != 0u;
            }
            u32 lincl = links;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                u32 v = __shfl_up_sync(FULL, lincl, o);
                if (lane >= o) lincl += v;
            }
            const u32 ltotal = __shfl_sync(FULL, lincl, 31);
            if (tail + ltotal > p.cq_cap) return false;
            if (lane < n && links) {
                u32 at = tail + lincl - links;
                const int cn = (int)size - HDR;
                for (int j = 0; j < cn; ++j)
                    if (EDGE_CHILD(slab[src + HDR + j].w) != 0u) q[at++] = (nu << 8) | (u32)j;
            }
            tail += ltotal;
            alloc += total;
            if (!root_step) head += (u32)n;
            root_step = false;
            __syncwarp();
            if (head >= tail) break;
        }
        out_units = alloc;
        return true;
    }

    // ---- the decision node's statistics and position, recorded when a move is made ----
    __device__ void record_root(const H& h, const P& pos, int n, size_t ri) {
        uint4 dummy = slab[0];
        for (int i = lane; i < G::ACTIONS; i += 32) sm.pol[i] = 0.0f;
        __syncwarp();
        for (int base = 0; base < n; base += 32) {
            int k = base + lane;
            if (k < n) {
                uint4 e = slab[ROOT_UNIT + HDR + k];
                int a = (int)EDGE_ACTION(e.w);
                sm.pol[a] = __uint_as_float(e.z);
                if (p.record_stats) {
                    p.rec_N[ri * G::ACTIONS + a] = __uint_as_float(e.z);
                    p.rec_W[ri * G::ACTIONS + a] = __uint_as_float(e.y);
                    p.rec_P[ri * G::ACTIONS + a] = p.add_noise ? p.root_p[(size_t)tree * G::ACTIONS + k] : __uint_as_float(e.x);
                }
            }
        }
        __syncwarp();
        if (lane == 0) {
            if (p.record_stats) {
                p.rec_root_W[ri] = __uint_as_float(dummy.y);
                p.rec_root_N[ri] = __uint_as_float(dummy.z);
                p.rec_trav[ri] = st.traversals;
            }
            for (int w = 0; w < W; ++w) {
                p.rec_board[ri * 2 * W + w] = h.b0.word(w);
                p.rec_board[ri * 2 * W + W + w] = h.b1.word(w);
            }
            p.rec_player[ri] = (unsigned char)pos.player;
        }
    }

    // ---- UCTTree::advanceDecision (uct/UCTTree.hpp:197-210) to edge slot ksel of the decision node ----
    __device__ bool advance_root(const H& h, const P& pos, int ksel, int action) {
        const u32 edge_unit = ROOT_UNIT + HDR + ksel;
        uint4 es = slab[edge_unit];
        u32 child = EDGE_CHILD(es.w);
        float own_w = __uint_as_float(es.y), own_n = __uint_as_float(es.z);
        if (child == 0) {
            P cp;
            make_child_pos(pos, ROOT_UNIT, action, cp);
            u32 need = HDR + (cp.terminal ? 0u : (u32)cp.n_legal());
            if (st.n_units + need + SLAB_SLACK > p.cap_units) { st.status = ST_ERR_CAPACITY; return false; }
            child = st.n_units;
            st.n_units += need;
            H ch;
            write_node(slab, child, cp, ROOT_UNIT, edge_unit, ch);
            own_w = (cfg_init_q() == SPRL_INITQ_PARENT && (h.meta & META_EVALUATED)) ? h.net_value : 0.0f;
            __syncwarp();
        }
        if (st.n_units > st.high_water) st.high_water = st.n_units;
        uint4* dst = slab_ptr(st.slab ^ 1u);
        u32 units = 0;
        if (!compact_into(dst, child, own_w, own_n, units)) { st.status = ST_ERR_CAPACITY; return false; }
        st.slab ^= 1u;
        slab = dst;
        st.n_units = units;
        st.traversals = 0;
        st.move_count += 1;
        st.n_queued = 0;
        __syncwarp();
        return true;
    }

    // ---- after a move: a finished game is recorded (`record`: once per game) and the slot starts its next one ----
    __device__ void after_move(bool record) {
        u32 rmeta = *HL<W>::meta_ptr(slab + ROOT_UNIT);
        if (META_TERMINAL(rmeta)) {
            // game over: the outcome of every recorded move is filled in by the sample writer
            if (lane == 0 && record) {
                p.rec_moves[st.game_index] = st.move_count - p.rec_open[st.game_index];
                p.rec_winner[st.game_index] = (unsigned char)META_WINNER(rmeta);
                p.rec_draws[st.game_index] = rng.ctr;
            }
            if (record) acc.games += 1;
            st.game_index += game_step;                  // static striding: game -> slot is deterministic
            if (st.game_index < p.iter->num_games) init_game();
            else { st.status = ST_DONE; }
        }
    }

    // ---- per-move finalisation of selfPlay (selfplay/SelfPlay.hpp:111-146) ----
    __device__ void finalize_move() {
        H h;
        HL<W>::load(slab + ROOT_UNIT, h);
        P pos;
        hdr_to_pos<G>(h, pos);
        const int n = META_NLEGAL(h.meta);
        if (st.move_count >= p.max_moves) { st.status = ST_ERR_MOVES; return; }
        const size_t ri = rec_index();
        record_root(h, pos, n, ri);             // leaves the visit counts in sm.pol
        // pdf = visits / sum; pdf = pow(pdf, e); pdf = pdf / sum; cdf = cumsum(pdf) / last
        float sum = 0.0f;
        for (int k = 0; k < n; ++k) sum += sm.pol[legal_action<G>(pos, k)];
        float inv = 1.0f / sum;
        const float ex = st.move_count - p.rec_open[st.game_index] < 15 ? 0.98f : 10.0f;   // constants.hpp:8-10; searched moves
        __syncwarp();
        for (int base = 0; base < n; base += 32) {
            int k = base + lane;
            if (k < n) { int a = legal_action<G>(pos, k); sm.pol[a] = det_powf(sm.pol[a] * inv, ex); }
        }
        __syncwarp();
        sum = 0.0f;
        for (int k = 0; k < n; ++k) sum += sm.pol[legal_action<G>(pos, k)];
        inv = 1.0f / sum;
        __syncwarp();
        for (int base = 0; base < n; base += 32) {
            int k = base + lane;
            if (k < n) { int a = legal_action<G>(pos, k); sm.pol[a] = sm.pol[a] * inv; }
        }
        __syncwarp();
        float run = 0.0f;
        for (int k = 0; k < n; ++k) {
            run = run + sm.pol[legal_action<G>(pos, k)];
            if (lane == 0) sm.aux[k] = run;
        }
        const float inv_last = 1.0f / run;
        __syncwarp();
        for (int i = lane; i < G::ACTIONS; i += 32) p.rec_pdf[ri * G::ACTIONS + i] = sm.pol[i];
        // Random::SampleCDF (utils/random.cpp:86-98)
        float e;
        do { e = rng_unit_f32(rng); } while (e == 0.0f);
        const float x = (run * inv_last) * e;
        int ksel = n - 1;
        for (int k = n - 1; k >= 0; --k) if (sm.aux[k] * inv_last >= x) ksel = k;
        const int action = legal_action<G>(pos, ksel);
        if (p.record_stats && lane == 0) p.rec_action[ri] = action;
        __syncwarp();
        if (!advance_root(h, pos, ksel, action)) return;
        acc.moves += 1;
        after_move(true);
    }

    // ---- UCTNetworkAgent::act after its search (agents/UCTNetworkAgent.hpp:59-105): the FIRST action with the
    //      most visits, then advanceDecision on the mover's own tree.  Returns the action (-1 on failure). ----
    __device__ int finalize_match_move() {
        H h;
        HL<W>::load(slab + ROOT_UNIT, h);
        P pos;
        hdr_to_pos<G>(h, pos);
        const int n = META_NLEGAL(h.meta);
        if (st.move_count >= p.max_moves) { st.status = ST_ERR_MOVES; return -1; }
        const size_t ri = rec_index();
        record_root(h, pos, n, ri);
        // std::max_element over all actions; illegal ones hold 0 visits.  (All-zero visit counts, possible only
        // when sims <= max_queue, make the reference play action 0 even when it is illegal; here the first legal one.)
        int ksel = 0;
        float best = -1.0f;
        for (int k = 0; k < n; ++k) {
            float v = sm.pol[legal_action<G>(pos, k)];
            if (v > best) { best = v; ksel = k; }
        }
        const int action = legal_action<G>(pos, ksel);
        if (p.record_stats && lane == 0) p.rec_action[ri] = action;
        __syncwarp();
        if (!advance_root(h, pos, ksel, action)) return -1;
        acc.moves += 1;
        after_move(true);
        return action;
    }

    // ---- IAgent::opponentAct (agents/UCTNetworkAgent.hpp:107-109): the other side's tree follows the move ----
    __device__ void follow_move(int action) {
        H h;
        HL<W>::load(slab + ROOT_UNIT, h);
        P pos;
        hdr_to_pos<G>(h, pos);
        if (!advance_root(h, pos, action_slot<G>(pos, action), action)) return;
        after_move(false);
    }

    // ---- UCTTree::advanceDecision(action) by the caller (uct/UCTTree.hpp:197-210), step-wise trees: the position is
    //      recorded (history of later network inputs, superko), the tree re-roots, a finished game stops the tree ----
    __device__ void caller_move(int action) {
        H h;
        HL<W>::load(slab + ROOT_UNIT, h);
        P pos;
        hdr_to_pos<G>(h, pos);
        const int n = META_NLEGAL(h.meta);
        const bool legal = !META_TERMINAL(h.meta) && action >= 0 &&
                           ((G::HAS_PASS && action == G::CELLS) ? pos.pass_legal != 0 : (action < G::CELLS && pos.legal.test(action)));
        if (!legal || st.n_queued > 0) { st.status = ST_ERR_ACTION; return; }
        if (st.move_count >= p.max_moves) { st.status = ST_ERR_MOVES; return; }
        const size_t ri = rec_index();
        record_root(h, pos, n, ri);
        if (p.record_stats && lane == 0) p.rec_action[ri] = action;
        for (int i = lane; i < G::ACTIONS; i += 32) p.rec_pdf[ri * G::ACTIONS + i] = 0.0f;     // no distribution: the caller chose
        __syncwarp();
        if (!advance_root(h, pos, action_slot<G>(pos, action), action)) return;
        acc.moves += 1;
        const u32 rmeta = *HL<W>::meta_ptr(slab + ROOT_UNIT);
        if (META_TERMINAL(rmeta)) {
            if (lane == 0) {
                p.rec_moves[st.game_index] = st.move_count - p.rec_open[st.game_index];
                p.rec_winner[st.game_index] = (unsigned char)META_WINNER(rmeta);
                p.rec_draws[st.game_index] = rng.ctr;
            }
            acc.games += 1;
            st.status = ST_DONE;
        }
    }
};

// ---- kernels -------------------------------------------------------------------------------------
constexpr int WARPS_PER_BLOCK = 1;          // 1: one tree per block, a finished tree frees its slot at once
constexpr int MIN_BLOCKS_PER_SM = 32;       // 32: 64 registers per thread -> 32 resident warps per SM

template <class G>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) k_begin(EngineParams p) {
    __shared__ WarpScratch scratch[WARPS_PER_BLOCK];
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= p.n_slots) return;
    TreeWarp<G> t(p, warp, lane, scratch[threadIdx.x >> 5]);
    t.st.game_index = warp;
    t.st.status = ST_IDLE;
    t.st.n_queued = 0;
    if (t.st.game_index < p.iter->num_games) { t.st.status = ST_PLAYING; t.init_game(); }
    else { t.st.status = ST_DONE; }
    t.save();
    if (lane == 0) {
        p.order[warp] = (u32)warp;
        if (warp == 0) { *p.order_parity = 0u; p.order_cnt[0] = p.order_cnt[1] = p.order_cnt[2] = p.order_cnt[3] = 0u; }
    }
}

// Lists `tree` for the next launch: front when it will finish a move there, back otherwise.
__device__ __forceinline__ void order_next(const EngineParams& p, u32 parity, int tree, bool heavy) {
    u32* cnt = p.order_cnt + (parity ^ 1u) * 2u;
    u32* dst = p.order + (size_t)(parity ^ 1u) * p.n_slots;
    if (heavy) dst[atomicAdd(cnt, 1u)] = (u32)tree;
    else dst[(u32)p.n_slots - 1u - atomicAdd(cnt + 1, 1u)] = (u32)tree;
}

// After every search launch: the list just written becomes current, the other one is emptied; the rows handed
// out by the launch become the evaluator's batch and the row counters restart.
__global__ void k_flip(EngineParams p) {
    p.q_rows[0] = p.q_count[0]; p.q_rows[1] = p.q_count[1];
    p.q_count[0] = 0u; p.q_count[1] = 0u;
    p.counters[3] = p.counters[2]; p.counters[2] = 0ULL;
    const u32 parity = *p.order_parity;
    p.order_cnt[parity * 2u] = 0u;
    p.order_cnt[parity * 2u + 1u] = 0u;
    *p.order_parity = parity ^ 1u;
}

template <class G>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MIN_BLOCKS_PER_SM) k_round(EngineParams p) {
    __shared__ WarpScratch scratch[WARPS_PER_BLOCK];
    const int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (slot >= p.n_slots) return;
    const u32 parity = *p.order_parity;
    const int warp = (int)p.order[(size_t)parity * p.n_slots + slot];        // the tree this warp serves
    if (p.trees[warp].status != ST_PLAYING) {
        if (lane == 0) order_next(p, parity, warp, false);
        return;
    }
    TreeWarp<G> t(p, warp, lane, scratch[threadIdx.x >> 5]);
    const bool stepwise = p.iter->stepwise != 0;
    const int sims = stepwise ? p.iter->step_sims : p.sims;
    bool waiting = false;                       // step-wise: the budget of the current move is spent, the caller moves
    for (int iter = 0; iter < p.rounds_per_launch; ++iter) {
        if (t.st.n_queued > 0) t.apply_leaves();
        if (t.st.traversals >= sims) {
            if (stepwise) { waiting = true; break; }
            t.finalize_move();
        }
        if (t.st.status != ST_PLAYING) break;
        t.search_batch();
        if (t.st.status != ST_PLAYING) break;
        if (p.evaluator == SPRL_EVAL_EXTERNAL || (stepwise && p.iter->step_single)) break;
    }
    if (t.st.status != ST_PLAYING && lane == 0) atomicAdd(&p.counters[t.st.status == ST_DONE ? 0 : 1], 1ULL);
    if (stepwise && !waiting && t.st.status == ST_PLAYING && lane == 0) atomicAdd(&p.counters[2], 1ULL);
    t.save();
    if (lane == 0) order_next(p, parity, warp, !stepwise && t.st.status == ST_PLAYING && t.st.traversals >= p.sims);
}

// ---- match play (Evaluate.cpp:93-157, evaluate/play.hpp:24-69): one warp per PAIR of trees ----
// The side to move searches in its own tree with its own evaluator; when its budget is spent it plays the
// most-visited action and both trees advance.  Game-level state (stream id and draw counter, move count, game
// index, status) is handed from one tree's record to the other's at every move; pair g's "side to move" lives in
// trees[g].pad.  Network k of game t plays Player (k ^ (t & 1)) (Evaluate.cpp:129-133).
template <class G>
__global__ void __launch_bounds__(32) k_match_begin(EngineParams p, MatchParams m) {
    __shared__ WarpScratch scratch;
    const int pair = blockIdx.x, lane = threadIdx.x;
    if (pair >= m.n_pairs) return;
    unsigned long long game_id = 0;
    u32 player = 0;
    for (int k = 0; k < 2; ++k) {
        TreeWarp<G, true> t(p, k * m.n_pairs + pair, lane, scratch, &p.iter->agent[k], m.n_pairs);
        t.st.game_index = pair;
        t.st.n_queued = 0;
        if (t.st.game_index < p.iter->num_games) { t.st.status = ST_PLAYING; t.init_game(); }
        else t.st.status = ST_DONE;
        game_id = t.st.game_id;
        player = META_PLAYER(*HL<G::W>::meta_ptr(t.slab + ROOT_UNIT));
        t.save();
    }
    __syncwarp();
    if (lane == 0) p.trees[pair].pad = player ^ (u32)(game_id & 1ULL);     // the side to move (ZERO, unless an opening line says otherwise)
}

template <class G>
__global__ void __launch_bounds__(32) k_match_round(EngineParams p, MatchParams m) {
    __shared__ WarpScratch scratch;
    const int pair = blockIdx.x, lane = threadIdx.x;
    if (pair >= m.n_pairs) return;
    if (p.trees[pair].status != ST_PLAYING) return;
    const int active = (int)p.trees[pair].pad;
    int action = -1, status, move_count;
    unsigned long long game_id, rng_ctr;
    long long game_index;
    {
        TreeWarp<G, true> t(p, active * m.n_pairs + pair, lane, scratch, &p.iter->agent[active], m.n_pairs);
        for (int iter = 0; iter < p.rounds_per_launch; ++iter) {
            if (t.st.n_queued > 0) t.apply_leaves();
            if (t.st.traversals >= p.sims) { action = t.finalize_match_move(); break; }
            t.search_batch();
            if (t.st.status != ST_PLAYING) break;
            if (t.cfg_evaluator() == SPRL_EVAL_EXTERNAL) break;
        }
        status = t.st.status; move_count = t.st.move_count; game_id = t.st.game_id; rng_ctr = t.rng.ctr;
        game_index = t.st.game_index;
        t.save();
    }
    if (action >= 0) {
        TreeWarp<G, true> o(p, (active ^ 1) * m.n_pairs + pair, lane, scratch, &p.iter->agent[active ^ 1], m.n_pairs);
        o.follow_move(action);                      // same position: same terminal test, same next game
        if (o.st.status == ST_ERR_CAPACITY) status = ST_ERR_CAPACITY;
        else { o.st.status = status; o.st.move_count = move_count; o.st.game_id = game_id; o.rng.game = game_id; o.rng.ctr = rng_ctr; o.st.game_index = game_index; }
        o.save();
        __syncwarp();
        if (status == ST_PLAYING && lane == 0) {
            const u32 player = META_PLAYER(*HL<G::W>::meta_ptr(o.slab + ROOT_UNIT));
            p.trees[pair].pad = player ^ (u32)(game_id & 1ULL);
        }
    }
    if (status != ST_PLAYING && lane == 0) {
        p.trees[pair].status = status;
        p.trees[m.n_pairs + pair].status = status;
        atomicAdd(&p.counters[status == ST_DONE ? 0 : 1], 1ULL);
    }
}

// ---- step-wise trees: the decision node's edge statistics (getDecisionNode()->getEdgeStatistics(), uct/UCTNode.hpp:45-60)
//      as dense [A] rows, and advanceDecision by the caller's action ----
template <class G>
__global__ void __launch_bounds__(32) k_tree_stats(EngineParams p, int n_trees, float* __restrict__ N, float* __restrict__ Wt, float* __restrict__ P,
                                                   float* __restrict__ root_N, float* __restrict__ root_W, signed char* __restrict__ player,
                                                   signed char* __restrict__ terminal, signed char* __restrict__ winner,
                                                   int* __restrict__ traversals, signed char* __restrict__ mask, int* __restrict__ queued) {
    const int tree = blockIdx.x, lane = threadIdx.x;
    if (tree >= n_trees) return;
    const TreeState& g = p.trees[tree];
    const uint4* slab = p.pool + ((size_t)tree * 2 + g.slab) * p.cap_units;
    constexpr int HDR = HL<G::W>::HDR;
    Hdr<G::W> h;
    HL<G::W>::load(slab + ROOT_UNIT, h);
    const int n = META_NLEGAL(h.meta);
    const bool expanded = (h.meta & META_EXPANDED) != 0;
    for (int i = lane; i < G::ACTIONS; i += 32) {
        const size_t at = (size_t)tree * G::ACTIONS + i;
        if (N) N[at] = 0.0f;
        if (Wt) Wt[at] = 0.0f;
        if (P) P[at] = 0.0f;
        if (mask) mask[at] = 0;
    }
    __syncwarp();
    for (int k = lane; k < n; k += 32) {
        const uint4 e = slab[ROOT_UNIT + HDR + k];
        const size_t at = (size_t)tree * G::ACTIONS + EDGE_ACTION(e.w);
        if (N) N[at] = __uint_as_float(e.z);
        if (Wt) Wt[at] = __uint_as_float(e.y);
        if (P) P[at] = !expanded ? 0.0f : (p.add_noise ? p.root_p[(size_t)tree * G::ACTIONS + k] : __uint_as_float(e.x));
        if (mask) mask[at] = 1;
    }
    if (lane == 0) {
        const uint4 d = slab[0];
        if (root_W) root_W[tree] = __uint_as_float(d.y);
        if (root_N) root_N[tree] = __uint_as_float(d.z);
        if (player) player[tree] = (signed char)META_PLAYER(h.meta);
        if (terminal) terminal[tree] = (signed char)META_TERMINAL(h.meta);
        if (winner) winner[tree] = (signed char)((int)META_WINNER(h.meta) - 1);      // device encoding: 0 none, 1 ZERO, 2 ONE
        if (traversals) traversals[tree] = g.traversals;
        if (queued) queued[tree] = g.n_queued;
    }
}

template <class G>
__global__ void __launch_bounds__(32) k_tree_advance(EngineParams p, int n_trees, const int* __restrict__ actions) {
    __shared__ WarpScratch scratch;
    const int tree = blockIdx.x, lane = threadIdx.x;
    if (tree >= n_trees) return;
    const int action = actions[tree];
    if (action < 0 || p.trees[tree].status != ST_PLAYING) return;      // -1: this tree stays where it is
    TreeWarp<G> t(p, tree, lane, scratch);
    t.caller_move(action);
    if (t.st.status != ST_PLAYING && lane == 0) atomicAdd(&p.counters[t.st.status == ST_DONE ? 0 : 1], 1ULL);
    t.save();
}

// ---- sample writer: selfPlay's symmetrised samples (selfplay/SelfPlay.hpp:86-96,127-136,
//      148-189) embedded as in runWorker (selfplay/GridWorker.hpp:146-196) ----
// One block per (game, move slot); writes S consecutive rows of states / distributions / outcomes.
template <class G>
__global__ void k_emit(EngineParams p, long long g0, const long long* __restrict__ game_row0, int S,
                       float* __restrict__ states, float* __restrict__ dists, float* __restrict__ outcomes) {
    constexpr int W = G::W, PLANES = 2 * G::HISTORY + 1, ROW = PLANES * G::CELLS;
    const long long g = g0 + blockIdx.x;    // grid = (games of the range, max_moves)
    if ((int)blockIdx.y >= p.rec_moves[g]) return;
    const int m = p.rec_open[g] + (int)blockIdx.y;     // searched move blockIdx.y; the opening's plies are history only
    const size_t ri = (size_t)g * p.max_moves + m;
    const int player = p.rec_player[ri];
    const unsigned char wn = p.rec_winner[g];
    const float outcome = (wn == WINNER_NONE) ? 0.0f : ((int)wn - 1 == player ? 1.0f : -1.0f);
    const long long row0 = game_row0[g] + (long long)blockIdx.y * S;
    // one thread per (symmetry, cell): the source cell is found once and serves every plane; a warp's
    // stores to a plane are contiguous
    for (int idx = threadIdx.x; idx < S * G::CELLS; idx += blockDim.x) {
        const int s = idx / G::CELLS, to = idx - s * G::CELLS;
        const int from = S > 1 ? sym_cell<G>(sym_inverse<G>(s), to) : to;
        const int w = from >> 6, sh = from & 63;
        float* out = states + (row0 + s) * ROW + to;
#pragma unroll
        for (int t = 0; t < G::HISTORY; ++t) {          // plane 2t: mover's stones, 2t+1: opponent's
            float mine = 0.0f, theirs = 0.0f;
            if (t <= m) {
                const unsigned long long* rb = p.rec_board + (ri - t) * 2 * W;
                mine = ((rb[player * W + w] >> sh) & 1ULL) ? 1.0f : 0.0f;
                theirs = ((rb[(1 - player) * W + w] >> sh) & 1ULL) ? 1.0f : 0.0f;
            }
            out[(2 * t) * G::CELLS] = mine;
            out[(2 * t + 1) * G::CELLS] = theirs;
        }
        out[(PLANES - 1) * G::CELLS] = player == 0 ? 1.0f : 0.0f;
        if constexpr (G::ACTIONS == G::CELLS + 1)        // placements move with their cells: new[f_s(i)] = old[i]
            dists[(row0 + s) * G::ACTIONS + to] = p.rec_pdf[ri * G::ACTIONS + from];
    }
    if constexpr (G::ACTIONS != G::CELLS + 1) {         // Connect Four: actions are columns
        for (int idx = threadIdx.x; idx < S * G::ACTIONS; idx += blockDim.x) {
            int s = idx / G::ACTIONS, j = idx - s * G::ACTIONS;
            int i = S > 1 ? sym_action<G>(sym_inverse<G>(s), j) : j;    // new[f_s(i)] = old[i]
            dists[(row0 + s) * G::ACTIONS + j] = p.rec_pdf[ri * G::ACTIONS + i];
        }
    } else if (threadIdx.x < S) {                        // the pass action maps to itself
        dists[(row0 + threadIdx.x) * G::ACTIONS + G::CELLS] = p.rec_pdf[ri * G::ACTIONS + G::CELLS];
    }
    if (threadIdx.x < S) outcomes[row0 + threadIdx.x] = outcome;
}

// ---- launchers used by engine.cu ---------------------------------------------------------------
template <class G> static void launch_begin(const EngineParams& p, cudaStream_t s) {
    k_begin<G><<<ceil_div(p.n_slots, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(p);
}
template <class G> static void launch_round(const EngineParams& p, cudaStream_t s) {
    k_round<G><<<ceil_div(p.n_slots, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(p);
    k_flip<<<1, 1, 0, s>>>(p);
}
template <class G> static void launch_emit(const EngineParams& p, long long g0, long long n_games, const long long* row0, int S, float* st,
                                           float* di, float* ou, cudaStream_t s) {
    k_emit<G><<<dim3((unsigned)n_games, (unsigned)p.max_moves), 256, 0, s>>>(p, g0, row0, S, st, di, ou);
}

template <class G> static void launch_tree_stats(const EngineParams& p, int n, float* N, float* W, float* P, float* rn, float* rw,
                                                 signed char* pl, signed char* te, signed char* wi, int* tr, signed char* mk, int* qu, cudaStream_t s) {
    k_tree_stats<G><<<n, 32, 0, s>>>(p, n, N, W, P, rn, rw, pl, te, wi, tr, mk, qu);
}
template <class G> static void launch_tree_advance(const EngineParams& p, int n, const int* actions, cudaStream_t s) {
    k_tree_advance<G><<<n, 32, 0, s>>>(p, n, actions);
}

template <class G> static void launch_match_begin(const EngineParams& p, const MatchParams& m, cudaStream_t s) {
    k_match_begin<G><<<m.n_pairs, 32, 0, s>>>(p, m);
}
template <class G> static void launch_match_round(const EngineParams& p, const MatchParams& m, cudaStream_t s) {
    k_match_round<G><<<m.n_pairs, 32, 0, s>>>(p, m);
    k_flip<<<1, 1, 0, s>>>(p);
}

#define GAME_SWITCH(game, STMT)                                   \
    switch (game) {                                               \
    case SPRL_GAME_OTHELLO: { typedef Othello G; STMT; break; }   \
    case SPRL_GAME_C4: { typedef ConnectFour G; STMT; break; }    \
    case SPRL_GAME_GO7: { typedef Go<7> G; STMT; break; }         \
    case SPRL_GAME_GO9: { typedef Go<9> G; STMT; break; }         \
    default: break;                                               \
    }

void search_launch_begin(int game, const EngineParams& p, cudaStream_t s) { GAME_SWITCH(game, launch_begin<G>(p, s)); }
void search_launch_round(int game, const EngineParams& p, cudaStream_t s) { GAME_SWITCH(game, launch_round<G>(p, s)); }
void search_launch_emit(int game, const EngineParams& p, long long g0, long long n_games, const long long* row0, int S, float* st, float* di,
                        float* ou, cudaStream_t s) { GAME_SWITCH(game, launch_emit<G>(p, g0, n_games, row0, S, st, di, ou, s)); }
void search_launch_match_begin(int game, const EngineParams& p, const MatchParams& m, cudaStream_t s) { GAME_SWITCH(game, launch_match_begin<G>(p, m, s)); }
void search_launch_match_round(int game, const EngineParams& p, const MatchParams& m, cudaStream_t s) { GAME_SWITCH(game, launch_match_round<G>(p, m, s)); }
void search_launch_tree_stats(int game, const EngineParams& p, int n, float* N, float* W, float* P, float* rn, float* rw, signed char* pl,
                              signed char* te, signed char* wi, int* tr, signed char* mk, int* qu, cudaStream_t s) {
    GAME_SWITCH(game, launch_tree_stats<G>(p, n, N, W, P, rn, rw, pl, te, wi, tr, mk, qu, s));
}
void search_launch_tree_advance(int game, const EngineParams& p, int n, const int* actions, cudaStream_t s) { GAME_SWITCH(game, launch_tree_advance<G>(p, n, actions, s)); }
int search_header_units(int game) { return (game == SPRL_GAME_GO9) ? 5 : 3; }

}  // namespace sprl
