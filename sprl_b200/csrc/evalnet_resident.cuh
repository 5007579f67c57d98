// evalnet_resident.cuh -- the evaluator tower with RESIDENT weights (included by evalnet.cu, namespace sprl::evalnet).
//
// Same network, same arithmetic and the same accumulation order as k_evalnet (evalnet.cu; the forward of
// /root/reference/src/networks/grid_networks.py:30-80 that /root/reference/cpp/src/networks/GridNetwork.hpp:99 runs),
// but the weights no longer stream from L2 for every tile.  k_evalnet re-reads 0.6 MB of split weights per 2-board
// tile (19.6 GB per 65,536-leaf launch for 1.2 MB of distinct bytes) and that stream shares the shared-memory port
// with the tensor cores' operand reads: the tensor pipe idles a third of the time.  Here
//
//   * the tower is cut into PHASES of at most one residual block (stem + block 1 | block 2 + heads for the 2-block
//     Othello / Connect Four nets); one launch per phase, every CTA keeps its phase's weights in shared memory for
//     the whole launch (loaded once, 150 KB), and the fp32 activations between phases go through HBM (32 KB per
//     tile, written and read once, in place);
//   * two CTAs of a cluster form a tcgen05 CTA PAIR (cta_group::2, M = 256): each CTA supplies its own 128-cell tile
//     and its own accumulators and holds HALF of the weight rows, which is what makes a whole block (2 x 147 KB of
//     hi/lo fp16 weights) fit the pair's shared memory, and halves the B-operand reads per SM;
//   * every CTA runs TWO tile streams (X, Y): own image pair, own 256 TMEM columns (192 accumulator + 64 residual),
//     own group of 8 epilogue warps.  The leader's MMA warp issues stage j of X, then of Y, then stage j+1 of X ...:
//     the epilogue of one stream runs under the MMAs of the other inside ONE CTA;
//   * the LAST stage of a phase never writes the image (its output goes to HBM or into the head convolutions), so its
//     epilogue also writes the NEXT tile's input (image + residual columns) channel group by channel group and the next
//     tile's first MMAs can be issued as soon as that epilogue ends; the 1x1 head convolutions (3 outputs) are 96 FMAs
//     per thread inside the last conv epilogue instead of an MMA stage of their own (which put two more barrier round
//     trips and the input load between two tiles: 4.5 k idle tensor cycles of 19 k per pair of tiles).
//
// Per SM and tile-layer the shared-memory port now carries 144 KB of A reads + 108 KB of B reads + 37 KB of image
// writes = 84 B/clk of 128 against 3.46 k cycles of MMAs (was: 147 + 221 + 147 KB of weight writes + 37).
//
// Shared memory per CTA: 4 images (2 streams x hi/lo) of 18,688 B -- the two zero rows above the first board row of a
// channel group double as the two zero rows below the last row of the previous group, so a group is 144 slots --
// then the resident weights, biases and 5 mbarriers: 229 KB for stem + block, 227 KB is the limit.
#pragma once

constexpr int RB_STREAMS = 2;
constexpr int RB_EPI_WARPS = 8;                              // per stream
constexpr int RB_MMA_WARP = RB_STREAMS * RB_EPI_WARPS;       // warp 16
constexpr int RB_THREADS = (RB_MMA_WARP + 1) * 32;           // 544
constexpr int RB_SLOTS = 144;                                // 16 zero slots + 128 cells; the next group's zero slots close this one
constexpr int RB_CG_STRIDE = RB_SLOTS * 16;                  // 2,304
constexpr int RB_IMG_BYTES = NCG * RB_CG_STRIDE + 256;       // 18,688 (+ the closing zero rows of the last group)
constexpr int RB_OFF_W = 2 * RB_STREAMS * RB_IMG_BYTES;      // 74,752
constexpr int RB_STREAM_COLS = 256;                          // TMEM columns of a stream: [0,192) accumulators, [192,256) residual
constexpr int RB_TMEM_COLS = RB_STREAMS * RB_STREAM_COLS;
constexpr int RB_MAX_STAGES = 4;
constexpr int RB_MAX_SMEM = 232448;
constexpr int RB_ACT_TILE_FLOATS = TILE_M * CH;              // fp32 activations of one tile between two phases

enum { RB_STEM = 0, RB_CONV = 1, RB_HEADS = 2 };
struct RbStage {
    int kind;          // RB_*
    int layer;         // index into NetDev::bias / inv_scale
    int ksteps;        // 16-channel k-steps per vertical tap
    int w_off;         // byte offset of the stage's weights in the CTA's resident region
    int add_res;       // second conv of a block: + block input (TMEM residual columns)
    int save_res;      // the output is the input of the block that follows in this phase
    int out_global;    // last stage of a phase that does not end the network: fp32 activations to HBM
    int heads;         // last conv of the network: the 1x1 head convolutions are computed from this stage's output
};
struct RbPhase {
    int n_stages;
    RbStage st[RB_MAX_STAGES];
    int in_planes_mode;          // 1: the input is the leaf planes (the phase starts with the stem); 0: `act`
    const unsigned char* w;      // [2][w_bytes]: the resident weights of CTA rank 0 / rank 1 (each holds half of the rows)
    int w_bytes;                 // per CTA, a multiple of 128
    float* act;                  // [tiles][16 channel quads][128 cells][4]: activations between phases, image units, in place
};
// linear lattice (boards wider than 8, one per tile): Z_-1 / Z_+1 of a warp's edge lanes for its neighbour warps,
// [stream][channel half][double buffer][warp of the quarter][left | right][16 values]
constexpr int RB_XCH_BYTES = RB_STREAMS * 2 * 2 * 4 * 2 * 16 * 4;
// fused head convolutions: fp32 weights [4][64] (rows above policy_channels are zero), then per stream the partial sums
// of the upper channel half, one float4 per cell
constexpr int RB_HEADW_BYTES = 4 * CH * 4;
constexpr int RB_HEADS_BYTES = RB_HEADW_BYTES + RB_STREAMS * TILE_M * 16;
__host__ __device__ inline int rb_smem_bytes(const RbPhase& ph, bool linear) {
    return RB_OFF_W + ph.w_bytes + ph.n_stages * CH * 4 + 64 + 16 + (linear ? RB_XCH_BYTES : 0) + (ph.st[ph.n_stages - 1].heads ? RB_HEADS_BYTES : 0);
}
__host__ __device__ inline int rb_stage_ndy(int kind) { return kind == RB_CONV ? 3 : 1; }
__host__ __device__ inline int rb_stage_n1(int kind) { return kind == RB_HEADS ? HEAD_N : 3 * CH; }
// bytes of a stage's weights held by ONE CTA of the pair: [dy][k chunk of 8][hi rows | lo rows of this CTA][8 halfs]
__host__ __device__ inline int rb_stage_bytes(int kind, int ksteps) { return rb_stage_ndy(kind) * ksteps * 2 * rb_stage_n1(kind) * 16; }

template <bool LINEAR>
__global__ void __launch_bounds__(RB_THREADS, 1)
k_evalnet_resident(NetDev net, RbPhase ph, const float* __restrict__ in, long long batch, const unsigned* __restrict__ d_rows) {
    extern __shared__ __align__(128) unsigned char smem[];
    if (d_rows) batch = min((long long)*d_rows, batch);          // batch size decided on the device by the search launch
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t s_base = smem_u32(smem);
    const int off_bias = RB_OFF_W + ph.w_bytes, off_bars = off_bias + ph.n_stages * CH * 4, off_tmem = off_bars + 64;
    const uint32_t bar_acc = s_base + off_bars;      // [2] accumulators of stream s complete (committed by the leader to both CTAs)
    const uint32_t bar_img = bar_acc + 16;           // [2] leader's copy is used: stream s's image is written and its accumulators
                                                     //     are drained in BOTH CTAs (one arrival per epilogue warp of the pair)
    const uint32_t bar_w = bar_img + 16;             // this CTA's resident weights have landed
    float* s_bias = reinterpret_cast<float*>(smem + off_bias);
    const long long n_tiles = LINEAR ? batch : (batch + 1) / 2, n_quads = (n_tiles + 3) / 4;      // a pair takes 4 tiles (2 streams x 2 CTAs) per turn
    const uint32_t crank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

    // ---- one-time setup ----
    for (int i = threadIdx.x; i < RB_OFF_W / 16; i += RB_THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = threadIdx.x; i < ph.n_stages * CH; i += RB_THREADS) {          // conv stages work in image units (x 2^ACT_SHIFT)
        const RbStage& S = ph.st[i / CH];
        s_bias[i] = net.bias[S.layer * CH + (i & (CH - 1))] * (S.kind != RB_HEADS ? ACT_SCALE : 1.0f);
    }
    const int off_heads = off_tmem + 16 + (LINEAR ? RB_XCH_BYTES : 0);
    if (ph.st[ph.n_stages - 1].heads)
        for (int i = threadIdx.x; i < 4 * CH; i += RB_THREADS)
            reinterpret_cast<float*>(smem + off_heads)[i] = i / CH <= net.policy_channels ? net.head_w[i] : 0.0f;
    if (threadIdx.x == 0) {
        for (int s = 0; s < RB_STREAMS; ++s) { mbar_init(bar_acc + 8 * s, 1); mbar_init(bar_img + 8 * s, 2 * RB_EPI_WARPS); }
        mbar_init(bar_w, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    proxy_fence();
    __syncthreads();
    cluster_sync_all();                               // the peer's barriers exist before anything arrives on them
    if (warp == RB_MMA_WARP) {                        // a collective of the two CTAs' MMA warps
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_base + off_tmem), "r"(RB_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        if (lane == 0) {                              // the phase's weights, once: this CTA's half of the rows
            mbar_expect_tx(bar_w, (uint32_t)ph.w_bytes);
            const unsigned char* src = ph.w + (size_t)crank * ph.w_bytes;
            for (int at = 0; at < ph.w_bytes; at += 16384)
                bulk_g2s(s_base + RB_OFF_W + at, src + at, (uint32_t)min(16384, ph.w_bytes - at), bar_w);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(smem + off_tmem), 0);

    if (warp == RB_MMA_WARP) {
        // ===== MMA issuer: the leader's warp runs the loop convergently, one elected lane issues =====
        if (crank == 0) {
            uint32_t img_phase = 0u;                                             // bit s: parity of stream s's next wait
            const bool split = net.single_pass == 0;                             // (SPRL_EVALNET_PRECISION_FP16: hi x hi only)
            constexpr uint32_t A_KSTEP = (2u * RB_CG_STRIDE) >> 4;
            for (long long quad = pair; quad < n_quads; quad += n_pairs) {
                for (int j = 0; j < ph.n_stages; ++j) {
                    const RbStage S = ph.st[j];
                    const int ndy = rb_stage_ndy(S.kind), n1 = rb_stage_n1(S.kind), nb = n1 / 2;   // nb weight rows per CTA
                    const uint32_t idesc = instr_desc_f16(2 * TILE_M, n1);
                    const uint32_t b_lbo = (uint32_t)(2 * nb) * 16u, b_kstep = (2u * b_lbo) >> 4, b_lo_off = ((uint32_t)nb * 16u) >> 4;
                    const uint64_t b0 = smem_desc(s_base + RB_OFF_W + S.w_off, b_lbo, 128);
#pragma unroll 1
                    for (int s = 0; s < RB_STREAMS; ++s) {
                        mbar_wait_cluster(bar_img + 8 * s, (img_phase >> s) & 1u, net.error_flag, 10 + s);
                        img_phase ^= 1u << s;
                        tc_fence_after();
                        const uint64_t a_hi0 = smem_desc(s_base + (2 * s) * RB_IMG_BYTES, RB_CG_STRIDE, 128);
                        const uint64_t a_lo0 = smem_desc(s_base + (2 * s + 1) * RB_IMG_BYTES, RB_CG_STRIDE, 128);
                        const uint32_t d_tmem = tmem + (uint32_t)(s * RB_STREAM_COLS);
                        uint32_t acc = 0;                                        // 0 for the stage's very first MMA only
                        for (int t = 0; t < ndy; ++t) {
                            // 16-byte slots: two storage rows per board row, or one row of `cols` cells in the linear lattice
                            const uint32_t a_off = (uint32_t)(16 + (LINEAR ? net.cols : 16) * (ndy == 3 ? t - 1 : 0));
                            const uint64_t bt = b0 + (uint32_t)(t * S.ksteps) * b_kstep;
#pragma unroll 2
                            for (int ks = 0; ks < S.ksteps; ++ks) {
                                const uint64_t ah = a_hi0 + a_off + ks * A_KSTEP, al = a_lo0 + a_off + ks * A_KSTEP, bd = bt + ks * b_kstep;
                                umma_f16_pair(d_tmem, ah, bd, idesc, acc);
                                if (split) {                                     // the two correction products of the hi/lo split
                                    umma_f16_pair(d_tmem, ah, bd + b_lo_off, idesc, 1u);
                                    umma_f16_pair(d_tmem, al, bd, idesc, 1u);
                                }
                                acc = 1;
                            }
                        }
                        umma_commit_pair(bar_acc + 8 * s);                      // both CTAs' epilogue groups of stream s
                        __syncwarp();
                    }
                }
            }
        }
    } else {
        // ===== epilogue group of stream s: cell m = TMEM lane m =====
        const int s = warp >> 3, w8 = warp & 7;
        const int m = (w8 & 3) * 32 + lane;                          // cell 0..127 = TMEM lane
        const int half = w8 >> 2;                                    // which half of the channels this warp finishes
        const int slot = cell_slot(m);
        const int g8 = m >> 3;
        const int r = LINEAR ? m / net.cols : g8 >> 1, c = LINEAR ? m - r * net.cols : m & 7, b = LINEAR ? 0 : g8 & 1;
        const bool valid = r < net.rows && c < net.cols;             // lattice positions outside the board stay zero
        const int cell = r * net.cols + c;
        // linear lattice: the left / right neighbour of lane 0 / 31 lives in another warp of the same stream and channel half
        const int wq = w8 & 3;
        float* xch = reinterpret_cast<float*>(smem + off_tmem + 16) + (s * 2 + half) * (2 * 4 * 2 * 16);
        const bool xl = LINEAR && lane == 0 && wq > 0, xr = LINEAR && lane == 31 && wq < 3;
        uint32_t xbuf = 0;
        const uint32_t t_lane = tmem + (uint32_t)(s * RB_STREAM_COLS) + ((uint32_t)((w8 & 3) * 32) << 16);
        uint4* a_hi = reinterpret_cast<uint4*>(smem + (2 * s) * RB_IMG_BYTES);
        uint4* a_lo = reinterpret_cast<uint4*>(smem + (2 * s + 1) * RB_IMG_BYTES);
        const uint32_t lead_img = map_to_cta(bar_img + 8 * s, 0);
        float mx = 0.0f;                                             // largest |image value| this thread produced
        const float vmask = valid ? 1.0f : 0.0f, lmask = c > 0 ? 1.0f : 0.0f, rmask = c + 1 < net.cols ? 1.0f : 0.0f;
        const int cells = net.rows * net.cols, planes = net.in_planes;
        uint32_t acc_phase = 0;
        // "my part of stream s's image is written and I am done reading its accumulators", to the leader's MMA warp
        auto signal = [&]() {
            proxy_fence();
            tc_fence_before();
            __syncwarp();
            // release at CTA scope: what was written is this CTA's own image, read by this CTA's tensor core (the pair's MMA
            // reads each tile from its own SM); the leader only learns that it may issue.  (A cluster-scope release costs a
            // MEMBAR.ALL.GPU per arrival -- 12 % of the epilogue's busy samples in the first ncu capture.)
            if (lane == 0) asm volatile("mbarrier.arrive.release.cta.shared::cluster.b64 _, [%0];" ::"r"(lead_img) : "memory");
        };
        // leaf planes -> stem image channels: channel dyi * planes + p of a cell holds plane p of the cell one row
        // above / at / below it (the stem's vertical taps are folded into K, see k_evalnet)
        auto load_planes = [&](long long tile_, int cg, float* v) {
            const long long board_ = LINEAR ? tile_ : tile_ * 2 + b;
#pragma unroll
            for (int j = 0; j < KCH; ++j) {
                const int ch = cg * KCH + j, dyi = ch / planes, p = ch - dyi * planes, rr = r + dyi - 1;
                v[j] = (valid && dyi < 3 && rr >= 0 && rr < net.rows && board_ < batch)
                           ? __ldg(in + (board_ * planes + p) * cells + rr * net.cols + c) : 0.0f;      // scaled at use: a prefetch must not wait for its data
            }
        };
        const int last_stage = ph.n_stages - 1;
        const long long quad_step = 4LL * n_pairs;
        const long long tile0 = (long long)pair * 4 + s * 2 + crank;
        const int xbar = 1 + s * 2 + half;                           // named barrier of this stream's channel half (4 warps)
        const int hbar = 5 + s * 4 + wq;                             // ... of the two warps that share a lane quarter (head sums)
        const float4* s_hw = reinterpret_cast<const float4*>(smem + off_heads);                       // [4][64]
        float4* s_hp = reinterpret_cast<float4*>(smem + off_heads + RB_HEADW_BYTES) + s * TILE_M;     // [cell]
        const bool planes_in = ph.in_planes_mode != 0;
        // stem image of a tile; its first channel group was prefetched into vnext
        float vnext[KCH];
        auto put_planes = [&](long long tile_) {
            for (int cg = half; cg < 2 * ph.st[0].ksteps; cg += 2) {
                float v[KCH];
                if (cg == half) {
#pragma unroll
                    for (int j = 0; j < KCH; ++j) v[j] = vnext[j] * ACT_SCALE;
                } else {
                    load_planes(tile_, cg, v);
#pragma unroll
                    for (int j = 0; j < KCH; ++j) v[j] *= ACT_SCALE;
                }
                uint4 h, l;
                split8(v, h, l, mx);
                a_hi[cg * RB_SLOTS + slot] = h;
                a_lo[cg * RB_SLOTS + slot] = l;
            }
        };
        // fp32 activations of the previous phase (image units), 16 channels of this thread's cell: residual columns + hi/lo image
        auto load_acts = [&](long long tile_, int q, float* x) {
            const float4* src = reinterpret_cast<const float4*>(ph.act) + (size_t)tile_ * (RB_ACT_TILE_FLOATS / 4) + m;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 t = tile_ < n_tiles ? __ldcg(src + (q * 4 + j) * TILE_M) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                x[4 * j] = t.x; x[4 * j + 1] = t.y; x[4 * j + 2] = t.z; x[4 * j + 3] = t.w;
            }
        };
        auto put_acts = [&](int q, const float* x) {
            tmem_st16(t_lane + RES_COL + q * 16, x);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                uint4 h, l;
                split8(x + KCH * j, h, l, mx);
                a_hi[(q * 2 + j) * RB_SLOTS + slot] = h;
                a_lo[(q * 2 + j) * RB_SLOTS + slot] = l;
            }
        };
        if (planes_in) load_planes(tile0, half, vnext);
        mbar_wait(bar_w, 0u, net.error_flag, 20);                   // (the leader's MMAs read both CTAs' weights: every arrival below implies them)
        float xin[16];
        // ---- input of the first tile; every later tile's input is written by the last stage's epilogue of the tile before ----
        if (planes_in) put_planes(tile0);
        else {
#pragma unroll 1
            for (int q = 2 * half; q < 2 * half + 2; ++q) { load_acts(tile0, q, xin); put_acts(q, xin); }
        }
        signal();
        for (long long tile = tile0; tile < n_quads * 4; tile += quad_step) {
            const long long board = LINEAR ? tile : tile * 2 + b;
            const long long next = tile + quad_step;
            const bool has_next = next < n_quads * 4;
            for (int j = 0; j <= last_stage; ++j) {
                const RbStage S = ph.st[j];
                const bool feed = j == last_stage && has_next;       // this epilogue also writes the next tile's input
                // accumulator -> image units; exact powers of two (read before the wait below, which hides the load)
                const float inv_scale = __ldg(net.inv_scale + S.layer) * ACT_SCALE;
                if (j == 0 && !planes_in && lane == 0 && next < n_tiles) {
                    // the next tile's activations towards L2, a whole tile ahead of their use
                    const float* nsrc = ph.act + (size_t)next * RB_ACT_TILE_FLOATS + (w8 & 3) * 32 * 4;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], 512;" ::"l"(nsrc + ((2 * half) * 4 + k) * TILE_M * 4) : "memory");
                }
                if (feed) {                                          // into registers under this stage's MMAs
                    if (planes_in) load_planes(next, half, vnext);
                    else load_acts(next, 2 * half, xin);
                }
                mbar_wait(bar_acc + 8 * s, acc_phase, net.error_flag, 30 + s);
                acc_phase ^= 1u;
                tc_fence_after();
                // the image is free from here on in the last stage: its MMAs are complete and its output does not go there
                if (feed && planes_in) put_planes(next);
                const float* bias = s_bias + j * CH;
                float hp0 = 0.0f, hp1 = 0.0f, hp2 = 0.0f;            // head convolutions over this thread's 32 channels
#pragma unroll 1
                for (int q = 2 * half; q < 2 * half + 2; ++q) {
                    // out[c] = Z_-1[c-1] + Z_0[c] + Z_+1[c+1]; Z_dx = accumulator columns [dx*64, dx*64+64)
                    float o[16], v[16], w[16];
                    tmem_ld16x3(t_lane + CH + q * 16, t_lane + q * 16, t_lane + 2 * CH + q * 16, o, v, w);   // dx = 0, -1, +1
                    if (LINEAR) {
                        // publish what the neighbouring warps need: lane 31's Z_-1 (for the next warp's lane 0) and lane 0's
                        // Z_+1 (for the previous warp's lane 31); double-buffered per iteration
                        float* mine = xch + (xbuf * 4 + wq) * 32;
                        if (lane == 31) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) mine[i] = v[i];
                        }
                        if (lane == 0) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) mine[16 + i] = w[i];
                        }
                        named_bar(xbar, 128);
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        float zl = __shfl_up_sync(0xffffffffu, v[i], 1), zr = __shfl_down_sync(0xffffffffu, w[i], 1);
                        if (xl) zl = xch[(xbuf * 4 + wq - 1) * 32 + i];
                        if (xr) zr = xch[(xbuf * 4 + wq + 1) * 32 + 16 + i];
                        o[i] = fmaf(zl, lmask, fmaf(zr, rmask, o[i]));
                    }
                    xbuf ^= 1u;
                    if (S.add_res) {                                                             // block input (image units), kept in TMEM
                        tmem_ld16(t_lane + RES_COL + q * 16, v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) o[i] = fmaxf(fmaf(o[i], inv_scale, v[i] + bias[q * 16 + i]), 0.0f) * vmask;
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) o[i] = fmaxf(fmaf(o[i], inv_scale, bias[q * 16 + i]), 0.0f) * vmask;
                    }
                    if (S.out_global) {
                        if (tile < n_tiles) {
                            float4* dst = reinterpret_cast<float4*>(ph.act) + (size_t)tile * (RB_ACT_TILE_FLOATS / 4) + m;
#pragma unroll
                            for (int jj = 0; jj < 4; ++jj)
                                __stcg(dst + (q * 4 + jj) * TILE_M, make_float4(o[4 * jj], o[4 * jj + 1], o[4 * jj + 2], o[4 * jj + 3]));
                        }
                    } else if (S.heads) {
                        // 1x1 head convolutions: rows 0..pc-1 policy conv, row pc value conv; ascending channel order
#pragma unroll
                        for (int i4 = 0; i4 < 4; ++i4) {
                            const float4 w0 = s_hw[q * 4 + i4], w1 = s_hw[16 + q * 4 + i4], w2 = s_hw[32 + q * 4 + i4];
                            hp0 = fmaf(o[4 * i4 + 3], w0.w, fmaf(o[4 * i4 + 2], w0.z, fmaf(o[4 * i4 + 1], w0.y, fmaf(o[4 * i4], w0.x, hp0))));
                            hp1 = fmaf(o[4 * i4 + 3], w1.w, fmaf(o[4 * i4 + 2], w1.z, fmaf(o[4 * i4 + 1], w1.y, fmaf(o[4 * i4], w1.x, hp1))));
                            hp2 = fmaf(o[4 * i4 + 3], w2.w, fmaf(o[4 * i4 + 2], w2.z, fmaf(o[4 * i4 + 1], w2.y, fmaf(o[4 * i4], w2.x, hp2))));
                        }
                    } else {
                        if (S.save_res) tmem_st16(t_lane + RES_COL + q * 16, o);
#pragma unroll
                        for (int jj = 0; jj < 2; ++jj) {
                            uint4 h, l;
                            split8(o + KCH * jj, h, l, mx);
                            a_hi[(q * 2 + jj) * RB_SLOTS + slot] = h;
                            a_lo[(q * 2 + jj) * RB_SLOTS + slot] = l;
                        }
                    }
                    if (feed && !planes_in) {
                        // this thread is done with residual columns q and the image is free: the next tile's channels q
                        put_acts(q, xin);
                        if (q == 2 * half) load_acts(next, q + 1, xin);
                    }
                }
                const bool heads_first = S.heads && last_stage == 0;     // (single-stage phase: the partial sums must be read before
                                                                         //  this warp lets the next tile's MMAs go)
                auto finish_heads = [&]() {
                    // upper channel half -> shared memory -> the warp of the lower half of the same cells; the ReLU'd
                    // activations go to HBM for k_heads
                    if (half == 1) {
                        s_hp[m] = make_float4(hp0, hp1, hp2, 0.0f);
                        __threadfence_block();
                        asm volatile("bar.arrive %0, 64;" ::"r"(hbar) : "memory");
                    } else {
                        named_bar(hbar, 64);
                        const float4 u = s_hp[m];
                        const int pc = net.policy_channels;
                        if (board < batch && valid) {
                            const float* hb = net.bias + (net.n_layers - 1) * CH;
                            float* dst = net.head_act + board * (long long)((pc + 1) * cells);
                            const float sum[3] = { hp0 + u.x, hp1 + u.y, hp2 + u.z };
#pragma unroll
                            for (int jj = 0; jj < 3; ++jj)
                                if (jj <= pc) dst[jj * cells + cell] = fmaxf(fmaf(sum[jj], 1.0f / ACT_SCALE, hb[jj]), 0.0f);
                        }
                    }
                };
                if (heads_first) finish_heads();
                if (j < last_stage || has_next) signal();
                if (S.heads && !heads_first) finish_heads();
            }
        }
        if (mx > HALF_MAX) atomicExch(net.error_flag + 1, 1ULL);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                               // no CTA leaves while its peer may still signal its barriers or read its tile
    if (warp == RB_MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(RB_TMEM_COLS) : "memory");
    }
}
