// games.cuh -- bitboard rules for the three games of the reference
// (/root/reference/cpp/src/games/{OthelloNode,ConnectFourNode,GoNode}.cpp).
//
// A position is two stone sets (player ZERO, player ONE), bit i = cell i in the
// reference's row-major indexing (row 0 on top).  Boards up to 64 cells use one
// 64-bit word per colour (Othello 8x8, Connect Four 7x6, Go 7x7); Go 9x9 uses two.
// Every game exposes the same static interface so that the environment kernels,
// the tree search and the sample writer are written once:
//
//   Game::start(Pos&)                      GameNode::setStartNodeImpl
//   Game::next(parent, action, hist, Pos&) GameNode::getNextNodeImpl
//
// `Pos` carries what the reference's GameNode carries: board, player to move,
// legal-action mask, terminal flag, winner (games/GameNode.hpp:192-200).
#pragma once
#include <cstdint>

namespace sprl {

typedef unsigned long long u64;
typedef unsigned int u32;

enum GameKind { GAME_OTHELLO = 0, GAME_C4 = 1, GAME_GO7 = 2, GAME_GO9 = 3 };
enum { WINNER_NONE = 0, WINNER_ZERO = 1, WINNER_ONE = 2 };

// ---- 1- and 2-word bit sets ---------------------------------------------------
template <int W> struct Bits;

template <> struct Bits<1> {
    u64 w0;
    __host__ __device__ Bits() : w0(0) {}
    __host__ __device__ explicit Bits(u64 a) : w0(a) {}
    __host__ __device__ static Bits bit(int i) { return Bits(1ULL << i); }
    __host__ __device__ bool test(int i) const { return (w0 >> i) & 1ULL; }
    __host__ __device__ bool any() const { return w0 != 0; }
    __host__ __device__ int count() const {
#ifdef __CUDA_ARCH__
        return __popcll(w0);
#else
        return __builtin_popcountll(w0);
#endif
    }
    __host__ __device__ Bits operator&(Bits o) const { return Bits(w0 & o.w0); }
    __host__ __device__ Bits operator|(Bits o) const { return Bits(w0 | o.w0); }
    __host__ __device__ Bits operator^(Bits o) const { return Bits(w0 ^ o.w0); }
    __host__ __device__ Bits operator~() const { return Bits(~w0); }
    __host__ __device__ bool operator==(Bits o) const { return w0 == o.w0; }
    __host__ __device__ bool operator!=(Bits o) const { return w0 != o.w0; }
    __host__ __device__ Bits shl(int n) const { return Bits(w0 << n); }
    __host__ __device__ Bits shr(int n) const { return Bits(w0 >> n); }
    __host__ __device__ u64 word(int) const { return w0; }
    __host__ __device__ void set_word(int, u64 v) { w0 = v; }
    // index of the lowest set bit (undefined when empty)
    __host__ __device__ int lowest() const {
#ifdef __CUDA_ARCH__
        return __ffsll((long long)w0) - 1;
#else
        return __builtin_ctzll(w0);
#endif
    }
    // number of set bits strictly below i
    __host__ __device__ int rank(int i) const { return Bits(w0 & ((1ULL << i) - 1ULL)).count(); }
};

template <> struct Bits<2> {
    u64 w0, w1;
    __host__ __device__ Bits() : w0(0), w1(0) {}
    __host__ __device__ Bits(u64 a, u64 b) : w0(a), w1(b) {}
    __host__ __device__ static Bits bit(int i) { return i < 64 ? Bits(1ULL << i, 0) : Bits(0, 1ULL << (i - 64)); }
    __host__ __device__ bool test(int i) const { return i < 64 ? ((w0 >> i) & 1ULL) : ((w1 >> (i - 64)) & 1ULL); }
    __host__ __device__ bool any() const { return (w0 | w1) != 0; }
    __host__ __device__ int count() const {
#ifdef __CUDA_ARCH__
        return __popcll(w0) + __popcll(w1);
#else
        return __builtin_popcountll(w0) + __builtin_popcountll(w1);
#endif
    }
    __host__ __device__ Bits operator&(Bits o) const { return Bits(w0 & o.w0, w1 & o.w1); }
    __host__ __device__ Bits operator|(Bits o) const { return Bits(w0 | o.w0, w1 | o.w1); }
    __host__ __device__ Bits operator^(Bits o) const { return Bits(w0 ^ o.w0, w1 ^ o.w1); }
    __host__ __device__ Bits operator~() const { return Bits(~w0, ~w1); }
    __host__ __device__ bool operator==(Bits o) const { return w0 == o.w0 && w1 == o.w1; }
    __host__ __device__ bool operator!=(Bits o) const { return !(*this == o); }
    __host__ __device__ Bits shl(int n) const { return Bits(w0 << n, (w1 << n) | (w0 >> (64 - n))); }  // 0 < n < 64
    __host__ __device__ Bits shr(int n) const { return Bits((w0 >> n) | (w1 << (64 - n)), w1 >> n); }
    __host__ __device__ u64 word(int i) const { return i ? w1 : w0; }
    __host__ __device__ void set_word(int i, u64 v) { if (i) w1 = v; else w0 = v; }
    __host__ __device__ int lowest() const {
#ifdef __CUDA_ARCH__
        return w0 ? __ffsll((long long)w0) - 1 : 64 + __ffsll((long long)w1) - 1;
#else
        return w0 ? __builtin_ctzll(w0) : 64 + __builtin_ctzll(w1);
#endif
    }
    __host__ __device__ int rank(int i) const {
        if (i < 64) return Bits<1>(w0).rank(i);
        return Bits<1>(w0).count() + (i == 64 ? 0 : Bits<1>(w1).rank(i - 64));
    }
};

// k-th (0-based) set bit of a 32-bit word by popcount bisection; k must be < popcount.
// (__fns is a software loop over the bits and dominated the search kernel's instruction count.)
__host__ __device__ __forceinline__ int nth_set_bit32(u32 x, int k) {
#ifdef __CUDA_ARCH__
    int r = 0, c;
    c = __popc(x & 0xffffu); if (k >= c) { k -= c; r += 16; x >>= 16; }
    c = __popc(x & 0xffu);   if (k >= c) { k -= c; r += 8;  x >>= 8; }
    c = __popc(x & 0xfu);    if (k >= c) { k -= c; r += 4;  x >>= 4; }
    c = __popc(x & 0x3u);    if (k >= c) { k -= c; r += 2;  x >>= 2; }
    c = (int)(x & 1u);       if (k >= c) { r += 1; }
    return r;
#else
    for (int i = 0; i < k; ++i) x &= x - 1;
    return __builtin_ctz(x);
#endif
}
// k-th (0-based) set bit of a 64-bit word; k must be < popcount.
__host__ __device__ __forceinline__ int nth_set_bit64(u64 x, int k) {
#ifdef __CUDA_ARCH__
    // one copy of the 32-bit bisection (the kernels inline this at ~30 sites: code size matters more than a select)
    const u32 lo = (u32)x, hi = (u32)(x >> 32);
    const int c = __popc(lo);
    const bool upper = k >= c;
    return (upper ? 32 : 0) + nth_set_bit32(upper ? hi : lo, upper ? k - c : k);
#else
    for (int i = 0; i < k; ++i) x &= x - 1;
    return __builtin_ctzll(x);
#endif
}
template <int W> __host__ __device__ inline int nth_set(const Bits<W>& b, int k);
template <> __host__ __device__ inline int nth_set<1>(const Bits<1>& b, int k) { return nth_set_bit64(b.w0, k); }
template <> __host__ __device__ inline int nth_set<2>(const Bits<2>& b, int k) {
    int c = Bits<1>(b.w0).count();
    return k < c ? nth_set_bit64(b.w0, k) : 64 + nth_set_bit64(b.w1, k - c);
}

// ---- generic position ----------------------------------------------------------
template <int W>
struct Pos {
    Bits<W> b[2];        // stones of player ZERO / ONE
    Bits<W> legal;       // legal non-pass actions (cells; columns for Connect Four)
    unsigned char player;      // 0 / 1 to move
    unsigned char pass_legal;  // the pass action (index CELLS) is legal
    unsigned char terminal;
    unsigned char winner;      // WINNER_*
    unsigned short depth;      // plies from the start position
    unsigned char action;      // action that led here (0 at the start position)
    __host__ __device__ int n_legal() const { return legal.count() + pass_legal; }
};

// History oracle handed to Game::next for rules that look at earlier positions
// (Go's positional superko).  Games without such rules ignore it.
// A history type answers seen(b0, b1) and enumerates its boards with for_each(f), f(b0, b1) -> void.
struct NoHistory {
    template <int W> __host__ __device__ bool seen(const Bits<W>&, const Bits<W>&) const { return false; }
    template <class F> __host__ __device__ void for_each(F&&) const {}
};

// a history with one more board in front of it
template <class Hist, int W>
struct HistPlus {
    const Hist& h;
    Bits<W> s0, s1;
    __host__ __device__ bool seen(const Bits<W>& a, const Bits<W>& b) const { return (a == s0 && b == s1) || h.seen(a, b); }
    template <class F> __host__ __device__ void for_each(F&& f) const { f(s0, s1); h.for_each(f); }
};

// ---- Othello (games/OthelloNode.cpp) ---------------------------------------------
struct Othello {
    static constexpr int W = 1, ROWS = 8, COLS = 8, CELLS = 64, ACTIONS = 65, HISTORY = 1, NSYM = 8;
    static constexpr int KIND = GAME_OTHELLO;
    static constexpr bool HAS_PASS = true;
    static constexpr int MAX_PLIES = 128;     // 60 placements, each followed by at most one pass
    typedef Pos<1> P;

    static constexpr u64 NOT_COL0 = 0xFEFEFEFEFEFEFEFEULL;   // cells with col != 0
    static constexpr u64 NOT_COL7 = 0x7F7F7F7F7F7F7F7FULL;   // cells with col != 7

    // one step of the whole set in direction d (order of games/OthelloNode.cpp:199-200)
    __host__ __device__ static u64 shift(u64 x, int d) {
        switch (d) {
        case 0: return x << 8;                   // ( 1, 0) south
        case 1: return (x << 9) & NOT_COL0;      // ( 1, 1)
        case 2: return (x << 1) & NOT_COL0;      // ( 0, 1) east
        case 3: return (x >> 7) & NOT_COL0;      // (-1, 1)
        case 4: return x >> 8;                   // (-1, 0) north
        case 5: return (x >> 9) & NOT_COL7;      // (-1,-1)
        case 6: return (x >> 1) & NOT_COL7;      // ( 0,-1) west
        default: return (x << 7) & NOT_COL7;     // ( 1,-1)
        }
    }

    // cells where `own` may place: empty, and some ray crosses >= 1 opponent stones
    // then reaches an own stone (canCapture, games/OthelloNode.cpp:226-252)
    __host__ __device__ static u64 mobility(u64 own, u64 opp) {
        u64 empty = ~(own | opp), moves = 0;
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            u64 t = shift(own, d) & opp;
#pragma unroll
            for (int i = 0; i < 5; ++i) t |= shift(t, d) & opp;
            moves |= shift(t, d) & empty;
        }
        return moves;
    }

    // stones turned by placing on `sq` (captures, games/OthelloNode.cpp:193-224)
    __host__ __device__ static u64 flips(u64 own, u64 opp, int sq) {
        u64 out = 0;
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            u64 x = shift(1ULL << sq, d), line = 0;
            while (x & opp) { line |= x; x = shift(x, d); }
            if (x & own) out |= line;
        }
        return out;
    }

#if defined(__CUDACC__) && (!defined(__CUDA_ARCH__) || __CUDA_ARCH__ >= 800)     // redux.sync: sm_80 and later
    // ---- warp-cooperative forms for kernels in which one warp owns a position (k_round): lane l walks
    //      direction l & 7 with per-lane shift amounts, branch-free, and the eight partial sets are OR-reduced
    //      by redux.sync.  All 32 lanes call with the same arguments and get the same result. ----
    struct LaneDir { int l, r; u64 keep; };
    __device__ static __forceinline__ LaneDir lane_dir(int lane) {
        const int d = lane & 7;
        const int amount = (0x71987198u >> (4 * d)) & 0xF;       // 8, 9, 1, 7, 8, 9, 1, 7
        const bool left = (0x87 >> d) & 1;                       // d = 0, 1, 2, 7 shift towards higher cells
        LaneDir k;
        k.l = left ? amount : 0;
        k.r = left ? 0 : amount;
        k.keep = ((0x0E >> d) & 1) ? NOT_COL0 : (((0xE0 >> d) & 1) ? NOT_COL7 : ~0ULL);
        return k;
    }
    __device__ static __forceinline__ u64 shift_lane(u64 x, const LaneDir& k) { return ((x << k.l) >> k.r) & k.keep; }
    __device__ static __forceinline__ u64 warp_or(u64 x) {
        const u32 lo = __reduce_or_sync(0xffffffffu, (u32)x), hi = __reduce_or_sync(0xffffffffu, (u32)(x >> 32));
        return ((u64)hi << 32) | lo;
    }
    __device__ static __forceinline__ u64 mobility_warp(u64 own, u64 opp, const LaneDir& k) {
        u64 t = shift_lane(own, k) & opp;
#pragma unroll
        for (int i = 0; i < 5; ++i) t |= shift_lane(t, k) & opp;
        return warp_or(shift_lane(t, k) & ~(own | opp));
    }
    __device__ static __forceinline__ u64 flips_warp(u64 own, u64 opp, int sq, const LaneDir& k) {
        u64 t = shift_lane(1ULL << sq, k) & opp;                 // the run of opponent stones next to sq
#pragma unroll
        for (int i = 0; i < 5; ++i) t |= shift_lane(t, k) & opp;
        return warp_or((shift_lane(t, k) & own) ? t : 0ULL);    // closed by an own stone
    }
    // next() with the direction loops spread over the lanes
    __device__ static void next_warp(const P& par, int action, int lane, P& p) {
        const LaneDir k = lane_dir(lane);
        u64 own = par.b[par.player].w0, opp = par.b[1 - par.player].w0;
        if (action != CELLS) {
            u64 f = flips_warp(own, opp, action, k);
            own |= f | (1ULL << action);
            opp &= ~f;
        }
        p.b[par.player] = Bits<1>(own);
        p.b[1 - par.player] = Bits<1>(opp);
        p.player = 1 - par.player;
        p.depth = par.depth + 1;
        p.action = (unsigned char)action;
        u64 m_new = mobility_warp(opp, own, k);
        p.legal = Bits<1>(m_new);
        p.pass_legal = (m_new == 0);
        p.terminal = (m_new == 0) && (mobility_warp(own, opp, k) == 0);
        p.winner = WINNER_NONE;
        if (p.terminal) {
            int c0 = p.b[0].count(), c1 = p.b[1].count();
            if (c0 > c1) p.winner = WINNER_ZERO;
            if (c1 > c0) p.winner = WINNER_ONE;
        }
    }
#endif

    __host__ __device__ static void set_mask(P& p) {          // actionMask, :156-177
        u64 m = mobility(p.b[p.player].w0, p.b[1 - p.player].w0);
        p.legal = Bits<1>(m);
        p.pass_legal = (m == 0);
    }

    __host__ __device__ static void start(P& p) {             // :18-32
        p.b[0] = Bits<1>((1ULL << 28) | (1ULL << 35));        // (3,4), (4,3) = ZERO
        p.b[1] = Bits<1>((1ULL << 27) | (1ULL << 36));        // (3,3), (4,4) = ONE
        p.player = 0; p.terminal = 0; p.winner = WINNER_NONE; p.depth = 0; p.action = 0;
        set_mask(p);
    }

    template <class Hist>
    __host__ __device__ static void next(const P& par, int action, const Hist&, P& p) {   // :34-87
        u64 own = par.b[par.player].w0, opp = par.b[1 - par.player].w0;
        if (action != CELLS) {
            u64 f = flips(own, opp, action);
            own |= f | (1ULL << action);
            opp &= ~f;
        }
        p.b[par.player] = Bits<1>(own);
        p.b[1 - par.player] = Bits<1>(opp);
        p.player = 1 - par.player;
        p.depth = par.depth + 1;
        p.action = (unsigned char)action;
        u64 m_new = mobility(opp, own);                        // side to move is the old opponent
        p.legal = Bits<1>(m_new);
        p.pass_legal = (m_new == 0);
        p.terminal = (m_new == 0) && (mobility(own, opp) == 0);   // isTerminal, :179-191
        p.winner = WINNER_NONE;
        if (p.terminal) {
            int c0 = p.b[0].count(), c1 = p.b[1].count();
            if (c0 > c1) p.winner = WINNER_ZERO;
            if (c1 > c0) p.winner = WINNER_ONE;
        }
    }
};

// ---- Connect Four (games/ConnectFourNode.cpp) --------------------------------------
struct ConnectFour {
    static constexpr int W = 1, ROWS = 6, COLS = 7, CELLS = 42, ACTIONS = 7, HISTORY = 1, NSYM = 2;
    static constexpr int KIND = GAME_C4;
    static constexpr bool HAS_PASS = false;
    static constexpr int MAX_PLIES = 42;
    typedef Pos<1> P;

    __host__ __device__ static void start(P& p) {             // :13-21
        p.b[0] = Bits<1>(0); p.b[1] = Bits<1>(0);
        p.legal = Bits<1>(0x7F);                              // actions are columns
        p.pass_legal = 0; p.player = 0; p.terminal = 0; p.winner = WINNER_NONE; p.depth = 0; p.action = 0;
    }

    // stones of `own` in line through (row, col) along (dr, dc), counting the stone itself
    __host__ __device__ static int run(u64 own, int row, int col, int dr, int dc) {
        int count = 1;
#pragma unroll
        for (int s = -1; s <= 1; s += 2) {
            int r = row + s * dr, c = col + s * dc;
            while (r >= 0 && r < ROWS && c >= 0 && c < COLS && ((own >> (r * COLS + c)) & 1ULL)) {
                ++count; r += s * dr; c += s * dc;
            }
        }
        return count;
    }

    template <class Hist>
    __host__ __device__ static void next(const P& par, int action, const Hist&, P& p) {   // :23-78
        u64 own = par.b[par.player].w0, opp = par.b[1 - par.player].w0, occ = own | opp;
        int col = action, row = ROWS - 1;                     // row 0 is the top row
        while (row >= 0 && ((occ >> (row * COLS + col)) & 1ULL)) --row;
        own |= 1ULL << (row * COLS + col);
        occ = own | opp;
        bool win = run(own, row, col, 0, 1) >= 4 || run(own, row, col, 1, 0) >= 4 ||     // checkWin, :135-217
                   run(own, row, col, 1, 1) >= 4 || run(own, row, col, 1, -1) >= 4;
        bool filled = (occ & 0x7FULL) == 0x7FULL;             // top row full
        p.b[par.player] = Bits<1>(own);
        p.b[1 - par.player] = Bits<1>(opp);
        p.player = 1 - par.player;
        p.depth = par.depth + 1;
        p.action = (unsigned char)action;
        p.terminal = win || filled;
        p.winner = win ? (par.player == 0 ? WINNER_ZERO : WINNER_ONE) : WINNER_NONE;
        p.legal = Bits<1>(p.terminal ? 0ULL : (~occ & 0x7FULL));   // terminal => empty mask, :70-72
        p.pass_legal = 0;
    }
};

// ---- Go (games/GoNode.cpp), N x N with N = 7 (one word) or 9 (two words) --------------
template <int N> struct GoWords { static constexpr int W = (N * N <= 64) ? 1 : 2; };

template <int N>
struct Go {
    static constexpr int W = GoWords<N>::W, ROWS = N, COLS = N, CELLS = N * N, ACTIONS = N * N + 1;
    static constexpr int HISTORY = 8, NSYM = 8;                // games/GoNode.hpp:19
    static constexpr int KIND = (N == 7) ? GAME_GO7 : GAME_GO9;
    static constexpr bool HAS_PASS = true;
    static constexpr int MAX_PLIES = 2 * N * N;                // GO_MAX_DEPTH, games/GoNode.hpp:22
    typedef Pos<W> P;
    typedef Bits<W> B;

    __host__ __device__ static B board_mask() {
        B m;
        for (int i = 0; i < W; ++i) {
            int lo = 64 * i, hi = CELLS - lo;
            m.set_word(i, hi >= 64 ? ~0ULL : (hi <= 0 ? 0ULL : ((1ULL << hi) - 1ULL)));
        }
        return m;
    }
    __host__ __device__ static B col_mask(int col) {           // all cells of one column
        B m;
        for (int r = 0; r < N; ++r) m = m | B::bit(r * N + col);
        return m;
    }
    // the 4-neighbourhood of a set (games/GoNode.hpp:92-104)
    __host__ __device__ static B neighbors(const B& x, const B& not_col0, const B& not_colN, const B& all) {
        return (x.shl(N) | x.shr(N) | (x.shl(1) & not_col0) | (x.shr(1) & not_colN)) & all;
    }

    struct Masks { B all, not_col0, not_colN; };
    __host__ __device__ static Masks masks() {
        Masks m;
        m.all = board_mask();
        m.not_col0 = m.all & ~col_mask(0);
        m.not_colN = m.all & ~col_mask(N - 1);
        return m;
    }

    // flood `seed` through `own`; returns the group
    __host__ __device__ static B flood(B seed, const B& own, const Masks& m) {
        B g = seed;
        for (;;) {
            B g2 = g | (neighbors(g, m.not_col0, m.not_colN, m.all) & own);
            if (g2 == g) return g;
            g = g2;
        }
    }

    // play `coord` for `own`; removes captured opponent groups (placePiece, games/GoNode.cpp:96-176)
    __host__ __device__ static void place(B& own, B& opp, int coord, const Masks& m) {
        B stone = B::bit(coord);
        own = own | stone;
        B adj = neighbors(stone, m.not_col0, m.not_colN, m.all) & opp;
        B captured;
        while (adj.any()) {
            B g = flood(B::bit(adj.lowest()), opp, m);
            B libs = neighbors(g, m.not_col0, m.not_colN, m.all) & ~(own | opp);
            if (!libs.any()) captured = captured | g;
            adj = adj & ~g;
        }
        opp = opp & ~captured;
    }

    // checkLegalPlacement (games/GoNode.cpp:178-228) as a rule: empty point, the placed
    // stone's group keeps a liberty after captures, and the new board matches no earlier one.
    template <class Hist>
    __host__ __device__ static bool legal_at(const B& own, const B& opp, int player, int coord,
                                             const Masks& m, const Hist& hist) {
        if ((own | opp).test(coord)) return false;
        B o = own, e = opp;
        place(o, e, coord, m);
        B g = flood(B::bit(coord), o, m);
        if (!(neighbors(g, m.not_col0, m.not_colN, m.all) & ~(o | e)).any()) return false;
        return player == 0 ? !hist.seen(o, e) : !hist.seen(e, o);
    }

    // The legal placements of the side to move, all at once (the same rule as legal_at, cell by cell):
    //   * a point that captures (it is the last liberty of an adjacent opponent group) never is suicide; its new board
    //     depends on the capture, so the superko test is the full one (legal_at) -- few points, rarely;
    //   * any other empty point p is no suicide iff it has an empty neighbour or touches an own group that keeps a
    //     liberty besides p (a group with at least two liberties); its new board is the current one plus the stone, so
    //     it repeats an earlier board h exactly when h has the same opponent stones and the own stones plus ONE more:
    //     one pass over the history instead of one per point.
    // `groups(own)`: a callback that, for a colour's stones, ORs the liberties of its groups with >= 2 liberties into
    // `multi` and the single liberties of its groups in atari into `atari` -- serial here, lane-parallel in the search.
    template <class Hist>
    __host__ __device__ static B legal_from_groups(const B& own, const B& opp, int player, const Masks& m, const Hist& hist,
                                                   const B& own_multi, const B& opp_atari) {
        const B empty = m.all & ~(own | opp);
        const B open = neighbors(empty, m.not_col0, m.not_colN, m.all);           // points with an empty neighbour
        const B capturing = empty & opp_atari;
        B plain = empty & ~capturing & (open | own_multi);
        if (plain.any()) {
            B repeats;
            hist.for_each([&](const B& h0, const B& h1) {
                const B& ho = player == 0 ? h0 : h1;
                const B& he = player == 0 ? h1 : h0;
                if (he == opp && (ho & own) == own) {
                    const B extra = ho ^ own;
                    if (extra.count() == 1) repeats = repeats | extra;
                }
            });
            plain = plain & ~repeats;
        }
        B legal = plain;
        for (B rest = capturing; rest.any();) {
            const int c = rest.lowest();
            rest = rest & ~B::bit(c);
            if (legal_at(own, opp, player, c, m, hist)) legal = legal | B::bit(c);
        }
        return legal;
    }
    // liberties of the groups of `stones`: >= 2 liberties -> multi, exactly one -> atari (`from`: the stones to start floods from)
    __host__ __device__ static void group_liberties(const B& from, const B& stones, const B& empty, const Masks& m, B& multi, B& atari) {
        for (B rest = from; rest.any();) {
            const B g = flood(B::bit(rest.lowest()), stones, m);
            const B libs = neighbors(g, m.not_col0, m.not_colN, m.all) & empty;
            const int n = libs.count();
            if (n >= 2) multi = multi | libs;
            else if (n == 1) atari = atari | libs;
            rest = rest & ~g;
        }
    }
    template <class Hist>
    __host__ __device__ static B legal_mask(const B& own, const B& opp, int player, const Masks& m, const Hist& hist) {
        const B empty = m.all & ~(own | opp);
        B own_multi, own_atari, opp_multi, opp_atari;
        group_liberties(own, own, empty, m, own_multi, own_atari);
        group_liberties(opp, opp, empty, m, opp_multi, opp_atari);
        return legal_from_groups(own, opp, player, m, hist, own_multi, opp_atari);
    }

    // Tromp-Taylor area count (countTerritory, games/GoNode.cpp:230-290)
    __host__ __device__ static void score(const B& b0, const B& b1, const Masks& m, int terr[2]) {
        terr[0] = b0.count(); terr[1] = b1.count();
        B empty = m.all & ~(b0 | b1);
        while (empty.any()) {
            B region = flood(B::bit(empty.lowest()), empty, m);
            B border = neighbors(region, m.not_col0, m.not_colN, m.all);
            bool t0 = (border & b0).any(), t1 = (border & b1).any();
            if (t0 && !t1) terr[0] += region.count();
            if (t1 && !t0) terr[1] += region.count();
            empty = empty & ~region;
        }
    }

    __host__ __device__ static float komi() { return N == 7 ? 9.0f : 7.5f; }   // games/GoNode.hpp:20, GoDesc.md:127-128

    __host__ __device__ static void start(P& p) {              // games/GoNode.cpp:303-317
        p.b[0] = B(); p.b[1] = B();
        p.legal = board_mask();
        p.pass_legal = 1; p.player = 0; p.terminal = 0; p.winner = WINNER_NONE; p.depth = 0; p.action = 0;
    }

    // The mask of the new position is NOT computed here (it needs the new node on
    // the history path and is the expensive part): callers run legal_at per cell,
    // possibly one lane per cell, and then set p.legal.
    template <class Hist>
    __host__ __device__ static void next_board(const P& par, int action, P& p) {   // games/GoNode.cpp:319-383
        const Masks m = masks();
        B own = par.b[par.player], opp = par.b[1 - par.player];
        if (action != CELLS) place(own, opp, action, m);
        p.b[par.player] = own;
        p.b[1 - par.player] = opp;
        p.player = 1 - par.player;
        p.depth = par.depth + 1;
        p.action = (unsigned char)action;
        // par.action is 0 at the start position, so it never counts as a pass there
        p.terminal = (par.depth > 0 && par.action == CELLS && action == CELLS) || p.depth >= MAX_PLIES;
        p.winner = WINNER_NONE;
        p.legal = B();
        p.pass_legal = p.terminal ? 0 : 1;                     // terminal => empty mask, :362-363
        if (p.terminal) {
            int terr[2];
            score(p.b[0], p.b[1], m, terr);
            float s0 = (float)terr[0], s1 = (float)terr[1];
            s1 += komi();
            if ((double)s0 > (double)s1 + 0.1) p.winner = WINNER_ZERO;
            else if ((double)s1 > (double)s0 + 0.1) p.winner = WINNER_ONE;
        }
    }

    // Single-thread version of the full transition (mask included).  `hist` must
    // answer for the boards of `par` and all its ancestors; the new board itself
    // cannot recur (a stone was added on an empty point).
    template <class Hist>
    __host__ __device__ static void next(const P& par, int action, const Hist& hist, P& p) {
        next_board<Hist>(par, action, p);
        if (p.terminal) return;
        const Masks m = masks();
        // the new node's own board and the parent's are ancestors of the new node's children as well
        const HistPlus<Hist, W> hs = { hist, p.b[0], p.b[1] };
        const HistPlus<HistPlus<Hist, W>, W> hp = { hs, par.b[0], par.b[1] };
        p.legal = legal_mask(p.b[p.player], p.b[1 - p.player], p.player, m, hp);
    }
};

// action index of the k-th legal action (ascending; the pass is last)
template <class G>
__host__ __device__ inline int legal_action(const typename G::P& p, int k) {
    int nc = p.legal.count();
    return k < nc ? nth_set<G::W>(p.legal, k) : G::CELLS;
}
// slot (rank) of a legal action
template <class G>
__host__ __device__ inline int action_slot(const typename G::P& p, int action) {
    return (G::HAS_PASS && action == G::CELLS) ? p.legal.count() : p.legal.rank(action);
}

// ---- compact position record: exchanged with the host (env.cu) and the opening table of the engine (search.cu) ----
struct alignas(16) PosRec {
    u64 b[4];       // b0 words, then b1 words (W each; unused = 0)
    u64 legal[2];
    int action;     // action | depth << 8 of the position (rollouts: the action taken from it)
    unsigned char player, pass_legal, terminal, winner;
    u32 parent;     // perft: index of the parent in the previous level
    u32 pad;
};

template <class G>
__host__ __device__ inline void pos_to_rec(const typename G::P& p, PosRec& r) {
    for (int i = 0; i < 2; ++i) {
        r.b[i] = i < G::W ? p.b[0].word(i) : 0;
        r.b[2 + i] = i < G::W ? p.b[1].word(i) : 0;
        r.legal[i] = i < G::W ? p.legal.word(i) : 0;
    }
    r.player = p.player; r.pass_legal = p.pass_legal; r.terminal = p.terminal; r.winner = p.winner;
    r.action = p.action | (p.depth << 8);   // perft keeps action/depth here; rollouts overwrite
    r.parent = 0; r.pad = 0;
}
template <class G>
__host__ __device__ inline void rec_to_pos(const PosRec& r, typename G::P& p) {
    for (int i = 0; i < G::W; ++i) {
        p.b[0].set_word(i, r.b[i]);
        p.b[1].set_word(i, r.b[2 + i]);
        p.legal.set_word(i, r.legal[i]);
    }
    p.player = r.player; p.pass_legal = r.pass_legal; p.terminal = r.terminal; p.winner = r.winner;
    p.action = (unsigned char)(r.action & 0xff); p.depth = (unsigned short)(r.action >> 8);
}

}  // namespace sprl
