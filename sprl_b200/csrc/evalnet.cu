// evalnet.cu -- the evaluator network's forward pass as one persistent tcgen05 kernel.
//
// Replaces, for boards up to 8x8 (Othello 8x8, Go 7x7, Connect Four 6x7; two boards per tile) and for boards of up to
// 128 cells in rows of at most 16 (Go 9x9; one board per tile), the LibTorch forward of the reference's traced
// `BasicGridNetwork` (/root/reference/cpp/src/networks/GridNetwork.hpp:99 calling the module
// of /root/reference/src/networks/grid_networks.py:30-80): conv3x3+BN+ReLU stem, `blocks`
// residual blocks of two conv3x3+BN, policy head (conv1x1 -> ReLU -> FC) and value head
// (conv1x1 -> ReLU -> FC -> ReLU -> FC -> tanh).  It reads the leaf planes the search kernel
// wrote (SPRL_EVAL_EXTERNAL buffers) and writes logits / value where the next search launch
// reads them.
//
// Design (B200, sm_100a):
//   * TWO CTAs per SM (each with half of the shared memory and 256 of the 512 TMEM columns), persistent
//     over tiles of TWO boards, each on an 8x8 lattice (smaller boards leave lattice positions zero)
//     = 128 cells = the M of one tcgen05.mma (cta_group::1, M=128).  A tile goes through the whole
//     tower on chip: activations never leave shared memory, fp32 accumulators live in TMEM.  Inside a
//     CTA the MMAs of a layer and its epilogue are serial (the next layer needs the whole image); the
//     second CTA fills the tensor pipe meanwhile, with no extra synchronisation.
//   * Every 3x3 convolution is an implicit GEMM with NO im2col copy.  The activation image is
//     kept in shared memory as [channel group of 8][storage row][8 cells][8 halfs], the rows of
//     the two boards interleaved and two zero rows above and below, so that a board row is one
//     128-byte, 128-byte-aligned UMMA core matrix (K-major, no swizzle: SBO = 128 B, LBO = one
//     channel group) and the operand of a tap with vertical offset dy is the SAME image with
//     the descriptor's start address moved by 2*dy storage rows.  Horizontal offsets are NOT
//     applied to the operand (a 16-byte shift would leave every core matrix straddling two
//     128-byte lines, measured 2x slower operand fetch): the taps of each dx accumulate into
//     their own TMEM accumulator Z_dx, and the epilogue forms out[c] = Z_-1[c-1] + Z_0[c] +
//     Z_+1[c+1] with two warp shuffles per value (cells of a board row are adjacent lanes).
//   * fp32 accuracy on the tensor cores by a two-term FP16 split: x = hi + lo with hi = fp16(x),
//     lo = fp16(x - hi); D = A_hi*W_hi + A_hi*W_lo + A_lo*W_hi, fp32 accumulate (products of fp16
//     operands are exact in fp32).  fp16 carries the same 11 significant bits as TF32, so the
//     split keeps ~22 bits like 3xTF32, but kind::f16 runs at twice the TF32 rate and K = 16 per
//     instruction halves the operand bytes.  fp16's narrow exponent is handled by exact
//     power-of-two scaling: activations are stored x 2^ACT_SHIFT (so their lo parts stay normal
//     down to 2^-7 and below that the absolute error is < 2^-29), each layer's weights x 2^s with
//     s chosen on the host so that max|W| lands in (2^9, 2^10], and the epilogue multiplies the
//     accumulator by 2^-(ACT_SHIFT + s).  Activations above 65504 / 2^ACT_SHIFT = 4094 would
//     overflow: they are clamped and reported (sprl_evalnet_status fails), never silently wrong.
//     (The reference evaluates in fp32; a single fp16/TF32 pass would lose 13 mantissa bits.)
//   * Weights (BN folded on the host in double, split hi/lo, pre-arranged as K-major UMMA
//     operands per tap, W_hi and W_lo stacked along N so that A_hi is read once for both) stream
//     from L2 through a ring of 24 KB units (32 input channels of one vertical offset) filled by
//     cp.async.bulk (multicast to the CTAs of a cluster) + mbarrier complete_tx; tcgen05.commit frees a unit.
//   * Warp roles: warps 0-7 = epilogue (TMEM -> registers -> shuffles/bias/residual/ReLU ->
//     hi/lo -> activation image; two warps per TMEM lane quarter, half of the channels each),
//     warp 8 = MMA issuer, warp 9 = weight producer.
//   * The stem (3 or 17 input planes) folds its three vertical taps into K (image channel dy * planes + p);
//     boards wider than 8 (Go 9x9) use the LINEAR lattice (k_evalnet<true>): one board per tile, cell
//     r * cols + c = TMEM lane, vertical taps = descriptor shifts by `cols` slots, and the left / right
//     neighbours that live in another warp are exchanged through a small shared-memory scratch.
//   * 128-channel towers (k_evalnet<., 128>): every conv layer is two output halves of 64 channels, each the same N = 192
//     MMA into its own accumulators; with the residual they take all 512 TMEM columns, so that instantiation runs one CTA
//     per SM.  The resident kernel has no room for their weights: they always take this kernel.
//   * A board's outputs do not depend on its row in the batch or on its tile partner (every CTA accumulates
//     in the same order), and the batch size may be read on the device (d_rows): the search kernel hands leaf
//     rows out by atomics and self-play stays reproducible.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_fp16.h>

#include "common.cuh"

namespace sprl {
namespace evalnet {

constexpr int TILE_M = 128;                  // cells per tile (two 8x8 boards)
constexpr int CH = 64;                       // tower width of the resident kernel and of the streaming kernel's output halves
constexpr int WIDE_CH = 128;                 // the other tower width the streaming kernel runs: two output halves of CH
constexpr int KCH = 8;                       // channels per 16-byte group (8 halfs)
constexpr int NCG = CH / KCH;                // channel groups
constexpr int KSTEP_CH = 2 * KCH;            // input channels per MMA (kind::f16: K = 16)
constexpr int ACT_SHIFT = 4;                 // activations are stored x 2^ACT_SHIFT in the fp16 images
constexpr float ACT_SCALE = 16.0f, HALF_MAX = 65504.0f;
constexpr int SLOTS = 160;                   // 20 storage rows x 8 cells
constexpr int CG_STRIDE = SLOTS * 16;        // bytes per channel group of the image
constexpr int UNIT_KS = 2;                   // k-steps (16 input channels each) per weight unit
constexpr int UNIT_BYTES = UNIT_KS * 2 * (6 * CH) * 16; // [K chunk of 8][3 dx x (hi, lo) x 64 rows][8 halfs]: 24 KB = 32 input channels of one dy
constexpr int MAX_NST = 12;                  // ring stages (as many as shared memory holds)
constexpr int MAX_LAYERS = 16;
// linear lattice: neighbours across a warp boundary are exchanged through shared memory,
// [channel half][double buffer][warp of the quarter][left / right][16 values]
constexpr int XCH_BYTES = 2 * 2 * 4 * 2 * 16 * 4;
constexpr int HEAD_N = 16;                   // policy channels (2) + value channel (1), padded
constexpr int EPI_WARPS = 8;                 // two warps per TMEM lane quarter, each takes half of the channels
constexpr int MMA_WARP = EPI_WARPS, PRODUCER_WARP = EPI_WARPS + 1;
constexpr int THREADS = (EPI_WARPS + 2) * 32;
constexpr int BAR1_THREADS = (EPI_WARPS + 1) * 32;   // epilogue warps + MMA warp
constexpr int CLUSTER = 2;                   // CTAs sharing one multicast weight stream
constexpr int RES_COL = 3 * CH;              // resident kernel: the block input of the current residual block, fp32, one cell per lane

// Streaming kernel (k_evalnet) geometry of a tower of C channels.  The C outputs of a conv layer are C / 64 output
// halves of 64 channels; every half is the same N = 192 MMA (3 dx x 64) into its own 192 TMEM columns
// [half * 192 + dx * 64 + channel], and the residual follows them: 64 channels use 256 columns, so two CTAs share an
// SM; 128 channels use all 512, so one CTA has the SM (its shared memory, 2 x 40 KB of image, holds ~5 ring stages).
template <int C> struct Width {
    static constexpr int NH = C / CH;                        // output halves
    static constexpr int IMG_BYTES = (C / KCH) * CG_STRIDE;  // 20,480 / 40,960
    static constexpr int TMEM_COLS = NH == 1 ? 256 : 512;
    static constexpr int RES_COL = 3 * CH * NH;              // the block input of the current residual block, fp32, one cell per lane
    static constexpr int CTAS_PER_SM = NH == 1 ? 2 : 1;      // resident CTAs per SM
    static constexpr int MAX_SMEM = (232448 - (CTAS_PER_SM - 1) * 1024) / CTAS_PER_SM;   // 227 KB per SM, 1 KB reserved per extra CTA
    static constexpr int CHUNKS = C / 32;                    // 16-channel epilogue chunks per warp (two warps per lane quarter)
    // shared memory map (bytes); the ring, the biases, the TMEM address (16 B), the linear lattice's neighbour scratch
    // and the barriers (full[nst], empty[nst], acc) follow at run-time offsets
    static constexpr int OFF_AHI = 0, OFF_ALO = IMG_BYTES, OFF_RING = 2 * IMG_BYTES;
    // TMEM column of accumulator dx = -1 for channels [16 q, 16 q + 16); dx = 0 and +1 follow at +64 and +128
    __device__ static constexpr int zcol(int q) { return q * 16 + (NH > 1 ? (q >> 2) * 2 * CH : 0); }
};
static_assert(Width<WIDE_CH>::RES_COL + WIDE_CH == Width<WIDE_CH>::TMEM_COLS, "128 channels fill the TMEM");

struct NetDev {
    const unsigned short* wunits;   // packed fp16 weight units in consumption order, `replicas` copies back to back
    long long wunits_bytes;  // bytes of one copy
    int replicas;
    const float* bias;       // [n_layers][channels]
    const float* pfc_wt;     // [128][actions]  (policy_fc.weight transposed)
    const float* pfc_b;      // [actions]
    const float* vfc1_wt;    // [cells][value_hidden] (value_fc1.weight transposed)
    const float* vfc1_b;     // [value_hidden]
    const float* vfc2_w;     // [value_hidden] weights, then the bias
    const float* head_w;     // [4][channels] fp32 weights of the 1x1 head convolutions (rows 0..pc-1 policy, row pc value, rest zero): k_evalnet_resident
    int n_layers;            // 1 stem + 2*blocks + 1 heads
    int rows, cols;          // board: cell (r, c) lives at lattice position (r, c) of an 8 x 8 tile half, or ...
    int linear;              // ... boards wider or taller than 8 (Go 9x9): ONE board per tile, cell r * cols + c = TMEM lane
    int in_planes;
    int in_ksteps;           // ceil(in_planes / 16)
    int actions;
    int policy_channels;     // 2
    int nst;                 // ring stages
    float* head_act;         // [batch][(policy_channels + 1) * 64]: ReLU'd 1x1-conv head activations, consumed by k_heads
    unsigned long long* error_flag;   // [0] pipeline barrier time-out, [1] an activation left the fp16-split range
    const float* inv_scale;  // [MAX_LAYERS] 2^-(ACT_SHIFT + weight shift of the layer): accumulator -> real units.  In device
                             // memory, not in this by-value struct: a captured CUDA graph must see the scales of update()
    int single_pass;         // SPRL_EVALNET_PRECISION_FP16 (resident kernel): one fp16 MMA per product instead of the three of the hi/lo split
};

template <int C> inline int smem_bytes_for(int n_layers, int nst) {
    return Width<C>::OFF_RING + nst * UNIT_BYTES + n_layers * C * 4 + 16 + XCH_BYTES + (2 * nst + 1) * 8;
}

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must end as a reported error, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, unsigned long long* error_flag, int where) {
    for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins) {
        if (spins > (1u << 26)) {
            if (error_flag) atomicExch(error_flag, 0xDEAD0000ULL | (unsigned)where);
            __trap();
        }
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// Slice of a weight unit to the same shared-memory offset of every CTA in the cluster; each
// destination's mbarrier (same CTA-relative offset) receives complete_tx for the slice.
__device__ __forceinline__ void bulk_g2s_multicast(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint16_t mask) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// One lane of a converged warp (elect.sync).  The issuing warp runs its loops convergently so that
// descriptors and addresses stay in uniform registers; only the issue itself is predicated.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (elect_one()) {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
                     ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    }
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if (elect_one()) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    }
}
// arrives on the mbarrier at the same offset in every CTA of `mask` once this CTA's MMAs retire
__device__ __forceinline__ void umma_commit_multicast(uint32_t bar, uint16_t mask) {
    if (elect_one()) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(bar), "h"(mask) : "memory");
    }
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (elect_one()) {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}"
                     ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    }
}
// arrives on the mbarrier at the same offset in both CTAs of the pair once the pair's MMAs retire
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    if (elect_one()) {
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(bar), "h"((uint16_t)3) : "memory");
    }
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// wait on a barrier the peer CTA arrives on
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity, unsigned long long* error_flag, int where) {
    for (uint32_t spins = 0; !mbar_try_wait_cluster(bar, parity); ++spins) {
        if (spins > (1u << 26)) {
            if (error_flag) atomicExch(error_flag, 0xDEAD0000ULL | (unsigned)where);
            __trap();
        }
    }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                   "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
                   "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
                   "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
                 : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// three 16-column loads of a lane's accumulators in flight at once, one wait
__device__ __forceinline__ void tmem_ld16x3(uint32_t ta, uint32_t tb, uint32_t tc, float* u, float* v, float* w) {
    uint32_t p[16], r[16], q[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(p[0]), "=r"(p[1]), "=r"(p[2]), "=r"(p[3]), "=r"(p[4]), "=r"(p[5]), "=r"(p[6]), "=r"(p[7]),
                   "=r"(p[8]), "=r"(p[9]), "=r"(p[10]), "=r"(p[11]), "=r"(p[12]), "=r"(p[13]), "=r"(p[14]), "=r"(p[15])
                 : "r"(ta) : "memory");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(tb) : "memory");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]),
                   "=r"(q[8]), "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15])
                 : "r"(tc) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) { u[i] = __uint_as_float(p[i]); v[i] = __uint_as_float(r[i]); w[i] = __uint_as_float(q[i]); }
}
// two floats -> packed fp16 pair (x0 in the low half), round to nearest, saturating at +-65504
__device__ __forceinline__ uint32_t pack_half2_sat(float x0, float x1) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(x1), "f"(x0));
    return r;
}
// Eight values already in image units (real value x 2^ACT_SHIFT) -> their fp16 hi and lo parts, one 16-byte
// channel group each.  `mx` tracks the largest magnitude seen: beyond 65504 the conversion saturates and the
// forward is reported as out of range.
__device__ __forceinline__ void split8(const float* x, uint4& hi, uint4& lo, float& mx) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float a = x[2 * j], b = x[2 * j + 1];
        mx = fmaxf(mx, fmaxf(fabsf(a), fabsf(b)));
        h[j] = pack_half2_sat(a, b);
        const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&h[j]));
        l[j] = pack_half2_sat(a - hf.x, b - hf.y);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}
// K-major, no swizzle: rows of a core matrix 16 B apart, 8-row groups SBO apart, K chunks (16 B) LBO apart
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lbo >> 4) & 0x3fffu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3fffu) << 32) | (1ULL << 46);
}
// kind::f16: D = fp32 (bit 4), A and B = fp16 (format 0), both K-major
__device__ __forceinline__ uint32_t instr_desc_f16(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// Layer geometry shared by the producer, the MMA issuer and the host packer.
// The three horizontal taps of a vertical offset dy read the SAME operand A (horizontal shifts are
// applied to the outputs, see the header), so their weights are stacked along N: one weight unit
// holds, for one dy and up to UNIT_KS k-steps, [K chunk of 8][rows][8 halfs] with rows =
// W_hi(dx=-1) | W_hi(0) | W_hi(+1) | W_lo(-1) | W_lo(0) | W_lo(+1), n rows each.  Per k-step three
// MMAs with N = 3n accumulate into the same columns [dx*n + channel]: A_hi*[W_hi x3], A_hi*[W_lo x3]
// and A_lo*[W_hi x3] -- each 4 KB read of A feeds 192 output columns.  The 1x1 head convolution is
// the same with one dx.  A conv layer of 128 channels is two such layers of 64 outputs over the same
// input, one after the other (`nh` output halves): all units of half 0, then all units of half 1.
struct LayerGeom { int ndy, ndx, ksteps, n, units_per_dy, nh; };
template <int C> __host__ __device__ inline LayerGeom layer_geom(int layer, int n_layers, int in_ksteps) {
    LayerGeom g;
    if (layer == 0) { g.ndy = 1; g.ndx = 3; g.ksteps = in_ksteps; g.n = CH; g.nh = C / CH; }      // stem: the three dy taps are folded into K
    else if (layer == n_layers - 1) { g.ndy = 1; g.ndx = 1; g.ksteps = C / KSTEP_CH; g.n = HEAD_N; g.nh = 1; }
    else { g.ndy = 3; g.ndx = 3; g.ksteps = C / KSTEP_CH; g.n = CH; g.nh = C / CH; }
    g.units_per_dy = (g.ksteps + UNIT_KS - 1) / UNIT_KS;
    return g;
}
__host__ __device__ inline int unit_ksteps(const LayerGeom& g, int u) { return g.ksteps - UNIT_KS * u < UNIT_KS ? g.ksteps - UNIT_KS * u : UNIT_KS; }
__host__ __device__ inline int unit_bytes(const LayerGeom& g, int u) { return unit_ksteps(g, u) * 2 * (2 * g.ndx * g.n) * 16; }

// slot of cell m (TMEM lane m) in the activation image: rows of the two boards interleaved,
// two zero rows first
__device__ __forceinline__ int cell_slot(int m) { return m + 16; }

template <bool LINEAR, int C>
__global__ void __launch_bounds__(THREADS, Width<C>::CTAS_PER_SM)
k_evalnet(NetDev net, const float* __restrict__ in, long long batch, const unsigned* __restrict__ d_rows,
          float* __restrict__ logits, float* __restrict__ value) {
    using W = Width<C>;
    extern __shared__ __align__(128) unsigned char smem[];
    if (d_rows) batch = min((long long)*d_rows, batch);          // batch size decided on the device by the previous kernel
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_layers = net.n_layers, nst = net.nst;
    const uint32_t s_base = smem_u32(smem);
    const int off_bias = W::OFF_RING + nst * UNIT_BYTES, off_tmem = off_bias + n_layers * C * 4, off_bars = off_tmem + 16 + XCH_BYTES;
    const uint32_t bar_full = s_base + off_bars, bar_empty = bar_full + nst * 8, bar_acc = bar_empty + nst * 8;
    float* s_bias = reinterpret_cast<float*>(smem + off_bias);
    const long long n_tiles = LINEAR ? batch : (batch + 1) / 2;
    // every CTA of a cluster walks the same number of tiles (the multicast ring is shared);
    // tiles past the end are dummies: zero input, no output
    const long long n_iters = (n_tiles + gridDim.x - 1) / gridDim.x;
    const long long tile_end = (long long)blockIdx.x + n_iters * gridDim.x;
    const uint32_t crank = cluster_ctarank();
    const int cluster_id = blockIdx.x / CLUSTER;
    constexpr uint16_t CMASK = (uint16_t)((1u << CLUSTER) - 1u);

    // ---- one-time setup ----
    for (int i = threadIdx.x; i < (2 * W::IMG_BYTES) / 16; i += THREADS)
        reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = threadIdx.x; i < n_layers * C; i += THREADS)           // conv layers work in image units (x 2^ACT_SHIFT)
        s_bias[i] = net.bias[i] * (i < (n_layers - 1) * C ? ACT_SCALE : 1.0f);
    if (threadIdx.x == 0) {
        for (int i = 0; i < nst; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, CLUSTER); }
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    proxy_fence();
    __syncthreads();
    cluster_sync_all();                               // peers' barriers exist before anything is multicast
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_base + off_tmem), "r"(W::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(smem + off_tmem), 0);

    if (warp == PRODUCER_WARP) {
        // ===== weight producer =====
        if (lane == 0) {
            uint32_t s = 0, ph = 0;
            for (long long tile = blockIdx.x; tile < tile_end; tile += gridDim.x) {
                // Every tile needs the whole 1.2 MB of weights (shared memory has no room to keep
                // them).  The CTAs of a cluster share ONE stream: each loads 1/CLUSTER of every unit
                // and multicasts it to all.  Clusters read different replicas so that the chip is not
                // pulling the same L2 lines at the same moment.  Every cluster walks the taps in the same
                // order: a board's accumulation order, and so its outputs, must not depend on its CTA.
                const unsigned char* layer_src = reinterpret_cast<const unsigned char*>(net.wunits) +
                                                 (size_t)(cluster_id % net.replicas) * net.wunits_bytes;
                for (int layer = 0; layer < n_layers; ++layer) {
                    const LayerGeom g = layer_geom<C>(layer, n_layers, net.in_ksteps);
                    int dy_bytes = 0;
                    for (int u = 0; u < g.units_per_dy; ++u) dy_bytes += unit_bytes(g, u);
                    for (int h = 0; h < g.nh; ++h) {                     // output halves (128 channels), one after the other
                        for (int t = 0; t < g.ndy; ++t) {
                            const unsigned char* src = layer_src + (size_t)t * dy_bytes;
                            for (int u = 0; u < g.units_per_dy; ++u) {
                                const uint32_t bytes = (uint32_t)unit_bytes(g, u);
                                mbar_wait(bar_empty + 8 * s, ph ^ 1u, net.error_flag, 1);
                                const uint32_t slice = bytes / CLUSTER;
                                mbar_expect_tx(bar_full + 8 * s, bytes);       // the whole unit: one slice from every CTA of the cluster
                                bulk_g2s_multicast(s_base + W::OFF_RING + s * UNIT_BYTES + crank * slice, src + crank * slice, slice,
                                                   bar_full + 8 * s, CMASK);
                                src += bytes;
                                if (++s == (uint32_t)nst) { s = 0; ph ^= 1u; }
                            }
                        }
                        layer_src += (size_t)g.ndy * dy_bytes;
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == MMA_WARP) {
        // ===== MMA issuer (the whole warp runs the loop; one elected lane issues) =====
        uint32_t s = 0, ph = 0;
        for (long long tile = blockIdx.x; tile < tile_end; tile += gridDim.x) {
            for (int layer = 0; layer < n_layers; ++layer) {
                const LayerGeom g = layer_geom<C>(layer, n_layers, net.in_ksteps);
                named_bar(1, BAR1_THREADS);                                      // the layer's input image is complete, the accumulators are drained
                tc_fence_after();
                const int n1 = g.ndx * g.n;                                      // output columns of one MMA = W_hi (and W_lo) rows of a unit
                const uint32_t idesc = instr_desc_f16(TILE_M, n1);
                const uint32_t b_lbo = (uint32_t)(2 * n1) * 16u, b_kstep = (2u * b_lbo) >> 4, b_lo_off = ((uint32_t)n1 * 16u) >> 4;
                const uint64_t a_hi0 = smem_desc(s_base + W::OFF_AHI, CG_STRIDE, 128), a_lo0 = smem_desc(s_base + W::OFF_ALO, CG_STRIDE, 128);
                const uint64_t b0 = smem_desc(s_base + W::OFF_RING, b_lbo, 128);
                constexpr uint32_t A_KSTEP = (2u * CG_STRIDE) >> 4;
                for (int h = 0; h < g.nh; ++h) {
                    const uint32_t d_main = tmem + h * 3 * CH;             // this half's accumulators
                    uint32_t acc = 0;                        // 0 for the very first MMA of the layer's half only
                    for (int t = 0; t < g.ndy; ++t) {                        // same order as the producer
                        const int dy = g.ndy == 3 ? t - 1 : 0;
                        // in 16-byte slots: two storage rows per board row, or one row of `cols` cells in the linear lattice
                        const uint32_t a_off = (uint32_t)(16 + (LINEAR ? net.cols : 16) * dy);
                        for (int u = 0; u < g.units_per_dy; ++u) {
                            const int nks = unit_ksteps(g, u);
                            mbar_wait(bar_full + 8 * s, ph, net.error_flag, 2);
                            tc_fence_after();
                            const uint64_t bd = b0 + s * (UNIT_BYTES >> 4);
                            const uint64_t ah = a_hi0 + a_off + (uint32_t)(UNIT_KS * u) * A_KSTEP, al = a_lo0 + a_off + (uint32_t)(UNIT_KS * u) * A_KSTEP;
                            if (nks == UNIT_KS) {
#pragma unroll
                                for (int ks = 0; ks < UNIT_KS; ++ks) {
                                    umma_f16(d_main, ah + ks * A_KSTEP, bd + ks * b_kstep, idesc, acc);
                                    umma_f16(d_main, ah + ks * A_KSTEP, bd + ks * b_kstep + b_lo_off, idesc, 1u);
                                    umma_f16(d_main, al + ks * A_KSTEP, bd + ks * b_kstep, idesc, 1u);
                                    acc = 1;
                                }
                            } else {
                                for (int ks = 0; ks < nks; ++ks) {
                                    umma_f16(d_main, ah + ks * A_KSTEP, bd + ks * b_kstep, idesc, acc);
                                    umma_f16(d_main, ah + ks * A_KSTEP, bd + ks * b_kstep + b_lo_off, idesc, 1u);
                                    umma_f16(d_main, al + ks * A_KSTEP, bd + ks * b_kstep, idesc, 1u);
                                    acc = 1;
                                }
                            }
                            umma_commit_multicast(bar_empty + 8 * s, CMASK);   // every CTA's producer learns that this CTA is done with the unit
                            if (++s == (uint32_t)nst) { s = 0; ph ^= 1u; }
                        }
                    }
                }
                umma_commit(bar_acc);                                  // the accumulators of this layer are complete
                __syncwarp();
            }
        }
    } else {
        // ===== epilogue warps: cell m = TMEM lane m =====
        const int m = (warp & 3) * 32 + lane;                        // cell 0..127 = TMEM lane
        const int half = warp >> 2;                                  // which half of the channels this warp finishes
        const int slot = cell_slot(m);
        const int g8 = m >> 3;
        const int r = LINEAR ? m / net.cols : g8 >> 1, c = LINEAR ? m - r * net.cols : m & 7, b = LINEAR ? 0 : g8 & 1;
        const bool valid = r < net.rows && c < net.cols;             // lattice positions outside the board stay zero
        // linear lattice: the left / right neighbour of lane 0 / 31 lives in another warp of the same channel half
        float* xch = reinterpret_cast<float*>(smem + off_tmem + 16) + half * (2 * 4 * 2 * 16);
        const int wq = warp & 3;
        const bool xl = LINEAR && lane == 0 && wq > 0, xr = LINEAR && lane == 31 && wq < 3;
        uint32_t xbuf = 0;
        const int cell = r * net.cols + c;
        const bool has_left = c > 0, has_right = c + 1 < net.cols;
        const uint32_t t_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint4* a_hi = reinterpret_cast<uint4*>(smem + W::OFF_AHI);
        uint4* a_lo = reinterpret_cast<uint4*>(smem + W::OFF_ALO);
        float mx = 0.0f;                                             // largest |image value| this thread produced
        const float vmask = valid ? 1.0f : 0.0f, lmask = has_left ? 1.0f : 0.0f, rmask = has_right ? 1.0f : 0.0f;
        const int cells = net.rows * net.cols, planes = net.in_planes;
        uint32_t acc_phase = 0;
        // ---- input planes -> image (the reference's planes are 0/1, but any fp32 input is split).  The stem
        // has few input planes, so its vertical taps are folded into K: image channel dyi * planes + p of a
        // cell holds plane p of the cell one row above / at / below it, and the stem becomes a single-dy layer
        // (3 MMAs per k-step instead of 9).
        auto load_planes = [&](long long tile_, int cg, float* v) {
            const long long board_ = LINEAR ? tile_ : tile_ * 2 + b;
#pragma unroll
            for (int j = 0; j < KCH; ++j) {
                const int ch = cg * KCH + j, dyi = ch / planes, p = ch - dyi * planes, rr = r + dyi - 1;
                v[j] = (valid && dyi < 3 && rr >= 0 && rr < net.rows && board_ < batch)
                           ? in[(board_ * planes + p) * cells + rr * net.cols + c] * ACT_SCALE : 0.0f;
            }
        };
        // the first channel group of the NEXT tile is fetched while this tile's head MMAs run (a global round trip per
        // tile otherwise sits between two tiles); further groups (Go: 51 stem channels) are loaded in place
        float vnext[KCH];
        load_planes(blockIdx.x, half, vnext);
        for (long long tile = blockIdx.x; tile < tile_end; tile += gridDim.x) {
            const long long board = LINEAR ? tile : tile * 2 + b;
            for (int cg = half; cg < 2 * net.in_ksteps; cg += EPI_WARPS / 4) {
                float v[KCH];
                if (cg == half) {
#pragma unroll
                    for (int j = 0; j < KCH; ++j) v[j] = vnext[j];
                } else {
                    load_planes(tile, cg, v);
                }
                uint4 h, l;
                split8(v, h, l, mx);
                a_hi[cg * SLOTS + slot] = h;
                a_lo[cg * SLOTS + slot] = l;
            }
            proxy_fence();
            for (int layer = 0; layer < n_layers; ++layer) {
                tc_fence_before();
                named_bar(1, BAR1_THREADS);
                if (layer == n_layers - 1 && tile + gridDim.x < tile_end) load_planes(tile + gridDim.x, half, vnext);
                // accumulator -> image units for the conv layers (real units for the heads); exact powers of two (read
                // before the wait below, which hides the load)
                const float inv_scale = __ldg(net.inv_scale + layer) * (layer < n_layers - 1 ? ACT_SCALE : 1.0f);
                mbar_wait(bar_acc, acc_phase, net.error_flag, 3);
                acc_phase ^= 1u;
                tc_fence_after();
                const float* bias = s_bias + layer * C;
                if (layer < n_layers - 1) {
                    const bool add_res = layer > 0 && (layer & 1) == 0;      // second conv of a block
                    const bool save_res = (layer & 1) == 0;                  // block input of the next block
#pragma unroll 1
                    for (int q = W::CHUNKS * half; q < W::CHUNKS * half + W::CHUNKS; ++q) {
                        // out[c] = Z_-1[c-1] + Z_0[c] + Z_+1[c+1]; Z_dx = hi half + lo half of accumulator dx
                        float o[16], v[16], w[16];
                        const int zc = W::zcol(q);
                        tmem_ld16x3(t_lane + CH + zc, t_lane + zc, t_lane + 2 * CH + zc, o, v, w);   // dx = 0, -1, +1
                        if (LINEAR) {
                            // publish what the neighbouring warps need: lane 31's Z_-1 (for the next warp's lane 0)
                            // and lane 0's Z_+1 (for the previous warp's lane 31); double-buffered per iteration
                            float* mine = xch + (xbuf * 4 + wq) * 32;
                            if (lane == 31) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) mine[i] = v[i];
                            }
                            if (lane == 0) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) mine[16 + i] = w[i];
                            }
                            if (half == 0) named_bar(2, 128); else named_bar(3, 128);   // constant ids: the kernel reserves 4 barriers
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            float zl = __shfl_up_sync(0xffffffffu, v[i], 1), zr = __shfl_down_sync(0xffffffffu, w[i], 1);
                            if (xl) zl = xch[(xbuf * 4 + wq - 1) * 32 + i];
                            if (xr) zr = xch[(xbuf * 4 + wq + 1) * 32 + 16 + i];
                            o[i] = fmaf(zl, lmask, fmaf(zr, rmask, o[i]));
                        }
                        xbuf ^= 1u;
                        if (add_res) {                                                               // block input (image units), kept in TMEM
                            tmem_ld16(t_lane + W::RES_COL + q * 16, v);
#pragma unroll
                            for (int i = 0; i < 16; ++i) o[i] = fmaxf(fmaf(o[i], inv_scale, v[i] + bias[q * 16 + i]), 0.0f) * vmask;
                        } else {
#pragma unroll
                            for (int i = 0; i < 16; ++i) o[i] = fmaxf(fmaf(o[i], inv_scale, bias[q * 16 + i]), 0.0f) * vmask;
                        }
                        if (save_res) tmem_st16(t_lane + W::RES_COL + q * 16, o);
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const int cg = q * 2 + j;
                            uint4 h, l;
                            split8(o + KCH * j, h, l, mx);
                            a_hi[cg * SLOTS + slot] = h;
                            a_lo[cg * SLOTS + slot] = l;
                        }
                    }
                    proxy_fence();
                } else {
                    // ---- heads (1x1): columns 0..pc-1 = policy conv channels, column pc = value conv.
                    // The ReLU'd activations go to global memory; the fully connected layers run in k_heads
                    // (they need 49 KB of weights that this kernel's shared memory has no room for).
                    float v[16];
                    tmem_ld16(t_lane, v);
                    const int pc = net.policy_channels;
                    if (board < batch && half == 0 && valid) {
                        float* dst = net.head_act + board * (long long)((pc + 1) * cells);
#pragma unroll
                        for (int j = 0; j < 3; ++j)
                            if (j <= pc) dst[j * cells + cell] = fmaxf(v[j] * inv_scale + bias[j], 0.0f);
                    }
                }
            }
        }
        if (mx > HALF_MAX) atomicExch(net.error_flag + 1, 1ULL);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                               // no CTA leaves while peers may still signal its barriers
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(W::TMEM_COLS) : "memory");
    }
}

#include "evalnet_resident.cuh"

// ---- heads: policy_fc and value_fc1/fc2 over the 1x1-conv activations k_evalnet left in HBM ----
// VH = the value head's hidden width (= the tower width).  HB boards per CTA step, weights staged once in shared memory,
// BPT boards x 4 outputs per thread: 64 boards with VH = 64, 32 with VH = 128 (its weights and hidden layer take twice
// the room, and 64 staged boards would not leave Go 9x9 with two policy channels within 227 KB).
template <int VH> struct Heads {
    static constexpr int HB = 64 * CH / VH;   // boards per CTA step
    static constexpr int BPT = HB / 16;       // boards per thread (16 board groups x 16 output groups)
};
constexpr int HP_STRIDE = 84;                 // policy weight row stride in floats (up to 82 actions, padded for float4 loads)

template <int VH>
__global__ void __launch_bounds__(256)
k_heads(NetDev net, long long batch, const unsigned* __restrict__ d_rows, float* __restrict__ logits, float* __restrict__ value) {
    constexpr int HB = Heads<VH>::HB, BPT = Heads<VH>::BPT;
    extern __shared__ __align__(16) float hs[];
    if (d_rows) batch = min((long long)*d_rows, batch);
    if ((long long)blockIdx.x * HB >= batch) return;
    const int pc = net.policy_channels, cells = net.rows * net.cols, K = pc * cells, A = net.actions, IN = (pc + 1) * cells;
    float* wp = hs;                           // [K][HP_STRIDE]
    float* wv = wp + K * HP_STRIDE;           // [cells][VH]
    float* xbuf = wv + cells * VH;            // [2][HB][IN]: the next HB boards arrive (cp.async) while these are computed
    float* hid = xbuf + 2 * HB * IN;          // [HB][VH + 1]
    float* wt = hid + HB * (VH + 1);          // [K]: weights of output 64 when it is the only one past 64 (the pass action)
    const bool lone_tail = A == 65;
    const int a_main = lone_tail ? 64 : A;
    const int t = threadIdx.x;
    // stages the activations of boards b0 .. b0+HB-1 into buffer `which` (rows past the batch are zero)
    auto stage = [&](long long b0, int which) {
        if (b0 < batch) {
            const int nb = (int)(batch - b0 < HB ? batch - b0 : HB);
            float* dst = xbuf + which * HB * IN;
            const float* src = net.head_act + b0 * IN;          // HB * IN floats per CTA step: 16-byte aligned
            const int n16 = nb * IN / 4;
            for (int i = t; i < n16; i += 256)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst + 4 * i)), "l"(src + 4 * i) : "memory");
            for (int i = 4 * n16 + t; i < HB * IN; i += 256) dst[i] = i < nb * IN ? src[i] : 0.0f;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    stage((long long)blockIdx.x * HB, 0);
    for (int i = t; i < K * HP_STRIDE; i += 256) { const int k = i / HP_STRIDE, a = i - k * HP_STRIDE; wp[i] = a < A ? net.pfc_wt[k * A + a] : 0.0f; }
    for (int i = t; i < cells * VH; i += 256) wv[i] = net.vfc1_wt[i];
    if (lone_tail) for (int k = t; k < K; k += 256) wt[k] = net.pfc_wt[k * A + 64];
    const int ag = t & 15, bg = t >> 4;       // 16 output groups x 16 board groups
    int cur = 0;
    for (long long b0 = (long long)blockIdx.x * HB; b0 < batch; b0 += (long long)gridDim.x * HB, cur ^= 1) {
        __syncthreads();                                         // everyone is done with the other buffer and with hid
        const int nb = (int)(batch - b0 < HB ? batch - b0 : HB);
        stage(b0 + (long long)gridDim.x * HB, cur ^ 1);          // prefetch the next step
        asm volatile("cp.async.wait_group 1;" ::: "memory");      // this step's rows have landed
        __syncthreads();
        const float* x = xbuf + cur * HB * IN;
        // policy_fc: outputs 4*ag .. 4*ag+3 for boards BPT*bg .. BPT*bg+BPT-1 (+ the outputs beyond 64, one per thread row)
        for (int a0 = 4 * ag; a0 < a_main; a0 += 64) {
            float acc[BPT][4];
#pragma unroll
            for (int i = 0; i < BPT; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
            // four k per step: one 128-bit read of every board's activations (IN and K are multiples of 4 or the tail
            // loop below takes over) against four 128-bit weight reads -> 8 shared-memory reads per 64 FMAs
            int k = 0;
            if ((IN & 3) == 0) {
                for (; k + 4 <= K; k += 4) {
                    float4 xv[BPT];
#pragma unroll
                    for (int i = 0; i < BPT; ++i) xv[i] = *reinterpret_cast<const float4*>(x + (BPT * bg + i) * IN + k);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const float4 w = *reinterpret_cast<const float4*>(wp + (k + kk) * HP_STRIDE + a0);
#pragma unroll
                        for (int i = 0; i < BPT; ++i) {
                            const float xs = kk == 0 ? xv[i].x : (kk == 1 ? xv[i].y : (kk == 2 ? xv[i].z : xv[i].w));
                            acc[i][0] = fmaf(xs, w.x, acc[i][0]); acc[i][1] = fmaf(xs, w.y, acc[i][1]);
                            acc[i][2] = fmaf(xs, w.z, acc[i][2]); acc[i][3] = fmaf(xs, w.w, acc[i][3]);
                        }
                    }
                }
            }
            for (; k < K; ++k) {
                const float4 w = *reinterpret_cast<const float4*>(wp + k * HP_STRIDE + a0);
#pragma unroll
                for (int i = 0; i < BPT; ++i) {
                    const float xv = x[(BPT * bg + i) * IN + k];
                    acc[i][0] = fmaf(xv, w.x, acc[i][0]); acc[i][1] = fmaf(xv, w.y, acc[i][1]);
                    acc[i][2] = fmaf(xv, w.z, acc[i][2]); acc[i][3] = fmaf(xv, w.w, acc[i][3]);
                }
            }
#pragma unroll
            for (int i = 0; i < BPT; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (BPT * bg + i < nb && a0 + j < A) logits[(b0 + BPT * bg + i) * A + a0 + j] = acc[i][j] + net.pfc_b[a0 + j];
        }
        if (lone_tail) {
            // Output 64 (Othello's pass) alone would cost the two lanes per warp that own outputs 0..3 a second full pass
            // over K, i.e. double the policy phase for every warp.  Instead each warp takes HB / 8 boards, the lanes split K
            // (stride 32, ascending) and a butterfly adds the 32 partial sums: the same order for every board.
            const int wid = t >> 5, ln = t & 31;
            for (int i = 0; i < HB / 8; ++i) {
                const int b = wid * (HB / 8) + i;
                float sacc = 0.0f;
                for (int k = ln; k < K; k += 32) sacc = fmaf(x[b * IN + k], wt[k], sacc);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
                if (ln == 0 && b < nb) logits[(b0 + b) * A + 64] = sacc + net.pfc_b[64];
            }
        }
        {   // value_fc1 + ReLU: outputs 64 * oh + 4*ag .. +3 for boards BPT*bg .. BPT*bg+BPT-1
            float acc[VH / 64][BPT][4];
#pragma unroll
            for (int oh = 0; oh < VH / 64; ++oh)
#pragma unroll
                for (int i = 0; i < BPT; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[oh][i][j] = 0.0f;
            int k = 0;
            if ((IN & 3) == 0 && (K & 3) == 0) {
                for (; k + 4 <= cells; k += 4) {
                    float4 xv[BPT];
#pragma unroll
                    for (int i = 0; i < BPT; ++i) xv[i] = *reinterpret_cast<const float4*>(x + (BPT * bg + i) * IN + K + k);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                        for (int oh = 0; oh < VH / 64; ++oh) {
                            const float4 w = *reinterpret_cast<const float4*>(wv + (k + kk) * VH + 64 * oh + 4 * ag);
#pragma unroll
                            for (int i = 0; i < BPT; ++i) {
                                const float xs = kk == 0 ? xv[i].x : (kk == 1 ? xv[i].y : (kk == 2 ? xv[i].z : xv[i].w));
                                acc[oh][i][0] = fmaf(xs, w.x, acc[oh][i][0]); acc[oh][i][1] = fmaf(xs, w.y, acc[oh][i][1]);
                                acc[oh][i][2] = fmaf(xs, w.z, acc[oh][i][2]); acc[oh][i][3] = fmaf(xs, w.w, acc[oh][i][3]);
                            }
                        }
                    }
                }
            }
            for (; k < cells; ++k) {
#pragma unroll
                for (int oh = 0; oh < VH / 64; ++oh) {
                    const float4 w = *reinterpret_cast<const float4*>(wv + k * VH + 64 * oh + 4 * ag);
#pragma unroll
                    for (int i = 0; i < BPT; ++i) {
                        const float xv = x[(BPT * bg + i) * IN + K + k];
                        acc[oh][i][0] = fmaf(xv, w.x, acc[oh][i][0]); acc[oh][i][1] = fmaf(xv, w.y, acc[oh][i][1]);
                        acc[oh][i][2] = fmaf(xv, w.z, acc[oh][i][2]); acc[oh][i][3] = fmaf(xv, w.w, acc[oh][i][3]);
                    }
                }
            }
#pragma unroll
            for (int oh = 0; oh < VH / 64; ++oh)
#pragma unroll
                for (int i = 0; i < BPT; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        hid[(BPT * bg + i) * (VH + 1) + 64 * oh + 4 * ag + j] = fmaxf(acc[oh][i][j] + net.vfc1_b[64 * oh + 4 * ag + j], 0.0f);
        }
        __syncthreads();
        if (t < nb) {   // value_fc2 + tanh
            float s = net.vfc2_w[VH];
            // same summation order for every board (its outputs must not depend on its row); rows of VH + 1 floats: no bank conflicts
            for (int j = 0; j < VH; ++j) s = fmaf(net.vfc2_w[j], hid[t * (VH + 1) + j], s);
            value[b0 + t] = tanhf(s);
        }
    }
}

template <int VH> static inline size_t heads_smem_bytes(int pc, int cells) {
    constexpr int HB = Heads<VH>::HB;
    return (size_t)(pc * cells * HP_STRIDE + cells * VH + 2 * HB * (pc + 1) * cells + HB * (VH + 1) + pc * cells) * sizeof(float);
}
static inline size_t heads_smem_bytes(int vh, int pc, int cells) {
    return vh == WIDE_CH ? heads_smem_bytes<WIDE_CH>(pc, cells) : heads_smem_bytes<CH>(pc, cells);
}

// ---- host: BN folding, hi/lo split, operand packing ------------------------------------------
// Power-of-two shift that brings the largest |w| of a layer into (2^9, 2^10]: fp16 keeps 11 significant bits
// of every weight down to 2^-13 of the largest one, and hi stays far below 65504.
static int weight_shift(const std::vector<std::vector<float>>& b) {
    float mx = 0.0f;
    for (const auto& v : b) for (float w : v) mx = std::max(mx, std::fabs(w));
    if (!(mx > 0.0f) || !std::isfinite(mx)) return 0;
    int e;
    std::frexp(mx, &e);                       // mx = f * 2^e, f in [0.5, 1)
    return std::max(-40, std::min(40, 10 - e));
}

// appends the units of one vertical offset: b[dx][n][k] (n < n_pad rows, k < kk), per unit of <= UNIT_KS*16
// input channels the layout [K chunk of 8][hi rows of every dx | lo rows of every dx][8 halfs]; weights x 2^shift
static void append_units(std::vector<unsigned short>& out, const std::vector<std::vector<float>>& b, int n_pad, int kk, int shift) {
    const int ndx = (int)b.size(), rows = ndx * n_pad;
    for (int k0 = 0; k0 < kk; k0 += UNIT_KS * KSTEP_CH)
        for (int kc = k0 / KCH; kc < std::min(kk, k0 + UNIT_KS * KSTEP_CH) / KCH; ++kc)
            for (int part = 0; part < 2; ++part)
                for (int r = 0; r < rows; ++r) {
                    const int dx = r / n_pad, n = r - dx * n_pad;
                    for (int j = 0; j < KCH; ++j) {
                        const float w = std::ldexp(b[dx][(size_t)n * kk + kc * KCH + j], shift);
                        const __half hi = __float2half_rn(w);
                        const __half v = part == 0 ? hi : __float2half_rn(w - __half2float(hi));
                        out.push_back(__half_as_ushort(v));
                    }
                }
}

// Resident format (k_evalnet_resident): the weights of one vertical offset held by CTA `h` of a pair,
// [K chunk of 8][hi rows | lo rows][8 halfs] over this CTA's half of the rows (row = dx * n_pad + n).
static void append_resident(std::vector<unsigned short>& out, const std::vector<std::vector<float>>& b, int n_pad, int kk, int shift, int h) {
    const int ndx = (int)b.size(), rows = ndx * n_pad, rows_per = rows / 2;
    for (int kc = 0; kc < kk / KCH; ++kc)
        for (int part = 0; part < 2; ++part)
            for (int r = h * rows_per; r < (h + 1) * rows_per; ++r) {
                const int dx = r / n_pad, n = r - dx * n_pad;
                for (int j = 0; j < KCH; ++j) {
                    const float w = std::ldexp(b[dx][(size_t)n * kk + kc * KCH + j], shift);
                    const __half hi = __float2half_rn(w);
                    const __half v = part == 0 ? hi : __float2half_rn(w - __half2float(hi));
                    out.push_back(__half_as_ushort(v));
                }
            }
}

// rows [h * CH, h * CH + CH) of the taps b[t0 .. t0 + n): the weights of output half h of a conv layer (see layer_geom)
static std::vector<std::vector<float>> output_half(const std::vector<std::vector<float>>& b, int t0, int n, int kk, int h) {
    std::vector<std::vector<float>> r;
    for (int t = t0; t < t0 + n; ++t) r.emplace_back(b[t].begin() + (size_t)h * CH * kk, b[t].begin() + (size_t)(h + 1) * CH * kk);
    return r;
}

// the streaming kernel's shared memory for a tower of `ch` channels, and the most one CTA of it may take
static int stream_smem_bytes(int ch, int n_layers, int nst) {
    return ch == WIDE_CH ? smem_bytes_for<WIDE_CH>(n_layers, nst) : smem_bytes_for<CH>(n_layers, nst);
}
static int stream_max_smem(int ch) { return ch == WIDE_CH ? Width<WIDE_CH>::MAX_SMEM : Width<CH>::MAX_SMEM; }

}  // namespace evalnet
}  // namespace sprl

using namespace sprl;
using namespace sprl::evalnet;

struct sprl_evalnet {
    int device = 0;
    int rows = 0, cols = 0, in_planes = 0, channels = 0, blocks = 0, actions = 0, policy_channels = 0, value_hidden = 0;
    NetDev dev;
    std::vector<void*> allocations;
    int sm_count = 0;
    uint64_t launches = 0;
    int64_t upload_bytes = 0;      // host -> device bytes of one weight load
    float* head_act = nullptr;     // [head_cap][(policy_channels + 1) * 64]
    int64_t head_cap = 0;
    // resident-weight path (k_evalnet_resident): one launch per phase, activations between phases in `act`
    std::vector<RbPhase> phases;   // empty: this network only runs on the streaming kernel
    const unsigned short* rb_weights = nullptr;
    float* act = nullptr;          // [act_cap_tiles][RB_ACT_TILE_FLOATS]
    int64_t act_cap_tiles = 0;
    int path = 0;                  // SPRL_EVALNET_PATH_*: 0 auto (resident when the network fits), 1 streaming, 2 resident
    int max_ctas = 0;              // SPRL_EVALNET_MAX_CTAS, read at create: caps the resident kernel's grid.  Set to 2, one CTA pair
                                   // walks every quad of the batch (the test of the pairs' quad loop); larger caps leave SMs to a
                                   // concurrent search launch (tools/explore_overlap.py)
    // First call allocates; later calls (a new generation's weights) overwrite in place, so device
    // pointers captured in a CUDA graph stay valid.
    template <typename T> int upload(const std::vector<T>& h, const T** out) {
        void* p = (void*)*out;
        cudaError_t err;
        if (!p) {
            err = cudaMalloc(&p, std::max<size_t>(h.size(), 1) * sizeof(T));
            if (err != cudaSuccess) return fail(SPRL_E_CAPACITY, "cudaMalloc failed: %s", cudaGetErrorString(err));
            allocations.push_back(p);
        }
        err = cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
        upload_bytes += (int64_t)(h.size() * sizeof(T));
        if (err != cudaSuccess) return fail(SPRL_E_CUDA, "cudaMemcpy failed: %s", cudaGetErrorString(err));
        *out = (const T*)p;
        return SPRL_OK;
    }
    void release() {
        for (void* p : allocations) cudaFree(p);
        allocations.clear();
        if (head_act) cudaFree(head_act);
        head_act = nullptr; head_cap = 0;
        if (act) cudaFree(act);
        act = nullptr; act_cap_tiles = 0;
        rb_weights = nullptr;
    }
};

static int check_conv(const sprl_conv_bn_params& c, const char* what) {
    if (!c.weight || !c.bias || !c.bn_weight || !c.bn_bias || !c.bn_mean || !c.bn_var)
        return fail(SPRL_E_INVALID, "null parameter pointer in %s", what);
    return SPRL_OK;
}

static int pack_and_upload(sprl_evalnet* e, const sprl_network_params* p) {
    const int C = p->channels, P = p->in_planes, L = 2 + 2 * p->blocks;
    const int in_k = KSTEP_CH * ((3 * P + KSTEP_CH - 1) / KSTEP_CH);      // stem input channels: (dy, plane), see k_evalnet
    const double eps = p->bn_eps > 0 ? p->bn_eps : 1e-5;
    std::vector<unsigned short> units;
    std::vector<float> bias((size_t)L * C, 0.0f), inv_scale(MAX_LAYERS, 0.0f);
    struct LayerW { std::vector<std::vector<float>> b; int n_pad, kk, shift; };       // b[dy * ndx + dx][n * kk + k], kept for the resident format
    std::vector<LayerW> layers;
    auto conv_layer = [&](const sprl_conv_bn_params& c, int cin, int kk, int layer) {
        std::vector<double> scale(C);
        for (int co = 0; co < C; ++co) {
            scale[co] = (double)c.bn_weight[co] / std::sqrt((double)c.bn_var[co] + eps);
            bias[(size_t)layer * C + co] = (float)(((double)c.bias[co] - (double)c.bn_mean[co]) * scale[co] + (double)c.bn_bias[co]);
        }
        std::vector<std::vector<float>> b(9, std::vector<float>((size_t)C * kk, 0.0f));      // [dy * 3 + dx]
        for (int t = 0; t < 9; ++t)
            for (int co = 0; co < C; ++co)
                for (int ci = 0; ci < cin; ++ci)
                    b[t][(size_t)co * kk + ci] = (float)((double)c.weight[((size_t)co * cin + ci) * 9 + t] * scale[co]);
        const int shift = weight_shift(b);            // one shift over all C outputs: both halves share the layer's inv_scale
        inv_scale[layer] = std::ldexp(1.0f, -(ACT_SHIFT + shift));
        for (int h = 0; h < C / CH; ++h)
            for (int dy = 0; dy < 3; ++dy) append_units(units, output_half(b, 3 * dy, 3, kk, h), CH, kk, shift);
        layers.push_back(LayerW{ std::move(b), C, kk, shift });
    };
    {   // stem: K index dy * P + plane, one unit group with the three dx stacked along N
        const sprl_conv_bn_params& c = p->stem;
        std::vector<std::vector<float>> b(3, std::vector<float>((size_t)C * in_k, 0.0f));
        for (int co = 0; co < C; ++co) {
            const double scale = (double)c.bn_weight[co] / std::sqrt((double)c.bn_var[co] + eps);
            bias[co] = (float)(((double)c.bias[co] - (double)c.bn_mean[co]) * scale + (double)c.bn_bias[co]);
            for (int ci = 0; ci < P; ++ci)
                for (int dy = 0; dy < 3; ++dy)
                    for (int dx = 0; dx < 3; ++dx)
                        b[dx][(size_t)co * in_k + dy * P + ci] = (float)((double)c.weight[((size_t)co * P + ci) * 9 + dy * 3 + dx] * scale);
        }
        const int shift = weight_shift(b);
        inv_scale[0] = std::ldexp(1.0f, -(ACT_SHIFT + shift));
        for (int h = 0; h < C / CH; ++h) append_units(units, output_half(b, 0, 3, in_k, h), CH, in_k, shift);
        layers.push_back(LayerW{ std::move(b), C, in_k, shift });
    }
    for (int i = 0; i < 2 * p->blocks; ++i) conv_layer(p->tower[i], C, C, 1 + i);
    {   // heads: rows 0..pc-1 policy_conv, row pc value_conv
        const int pc = p->policy_channels;
        std::vector<std::vector<float>> bb(1, std::vector<float>((size_t)HEAD_N * C, 0.0f));
        std::vector<float>& b = bb[0];
        for (int j = 0; j < pc; ++j) {
            for (int ci = 0; ci < C; ++ci) b[(size_t)j * C + ci] = p->policy_conv_w[(size_t)j * C + ci];
            bias[(size_t)(L - 1) * C + j] = p->policy_conv_b[j];
        }
        for (int ci = 0; ci < C; ++ci) b[(size_t)pc * C + ci] = p->value_conv_w[ci];
        bias[(size_t)(L - 1) * C + pc] = p->value_conv_b[0];
        const int shift = weight_shift(bb);
        inv_scale[L - 1] = std::ldexp(1.0f, -(ACT_SHIFT + shift));
        append_units(units, bb, HEAD_N, C, shift);
        layers.push_back(LayerW{ std::move(bb), HEAD_N, C, shift });
    }
    // ---- resident format: phases of [stem] [conv, conv] stage groups, as many per launch as shared memory holds; the
    // head convolutions ride on the network's last conv stage
    std::vector<RbPhase> phases;
    std::vector<unsigned short> rbw;
    std::vector<float> head_w(4 * (size_t)C, 0.0f);
    for (int j = 0; j <= p->policy_channels && j < 4; ++j)
        for (int ci = 0; ci < C; ++ci) head_w[(size_t)j * C + ci] = layers[L - 1].b[0][(size_t)j * C + ci];
    {
        const bool linear = p->rows > 8 || p->cols > 8;
        std::vector<std::vector<RbStage>> plan(1);
        auto plan_smem = [&](const std::vector<RbStage>& stages) {
            RbPhase t;
            memset(&t, 0, sizeof(t));
            t.n_stages = (int)stages.size();
            for (size_t j = 0; j < stages.size() && j < (size_t)RB_MAX_STAGES; ++j) { t.st[j] = stages[j]; t.w_bytes += rb_stage_bytes(stages[j].kind, stages[j].ksteps); }
            t.w_bytes = (t.w_bytes + 127) / 128 * 128;
            return rb_smem_bytes(t, linear);
        };
        auto add_group = [&](std::vector<RbStage> group) {
            std::vector<RbStage> both = plan.back();
            both.insert(both.end(), group.begin(), group.end());
            if (!plan.back().empty() && (both.size() > (size_t)RB_MAX_STAGES || plan_smem(both) > RB_MAX_SMEM)) plan.push_back(group);
            else plan.back() = both;
        };
        const int last_conv = L - 2;                              // layer index of the network's last conv (the stem if there are no blocks)
        add_group({ RbStage{ RB_STEM, 0, in_k / KSTEP_CH, 0, 0, 0, 0, last_conv == 0 ? 1 : 0 } });
        for (int b = 0; b < p->blocks; ++b)
            add_group({ RbStage{ RB_CONV, 1 + 2 * b, CH / KSTEP_CH, 0, 0, 0, 0, 0 },
                        RbStage{ RB_CONV, 2 + 2 * b, CH / KSTEP_CH, 0, 1, 0, 0, last_conv == 2 + 2 * b ? 1 : 0 } });
        // three head outputs: the fused head sums hold that many; 128 channels: one layer's weights alone exceed a CTA pair
        bool fits = C == CH && p->policy_channels <= 2;
        for (size_t i = 0; i < plan.size(); ++i) fits = fits && plan_smem(plan[i]) <= RB_MAX_SMEM;
        if (fits) {
            std::vector<size_t> w_at;                       // offset (in halfs) of every phase's [rank 0 | rank 1] weights
            for (size_t i = 0; i < plan.size(); ++i) {
                RbPhase ph;
                memset(&ph, 0, sizeof(ph));
                ph.n_stages = (int)plan[i].size();
                ph.in_planes_mode = plan[i][0].kind == RB_STEM ? 1 : 0;
                int off = 0;
                for (int j = 0; j < ph.n_stages; ++j) {
                    RbStage st = plan[i][j];
                    st.w_off = off;
                    off += rb_stage_bytes(st.kind, st.ksteps);
                    const bool last = j + 1 == ph.n_stages;
                    st.save_res = (!last && plan[i][j + 1].kind == RB_CONV && !plan[i][j + 1].add_res) ? 1 : 0;
                    st.out_global = (last && !st.heads) ? 1 : 0;
                    ph.st[j] = st;
                }
                ph.w_bytes = (off + 127) / 128 * 128;
                w_at.push_back(rbw.size());
                for (int h = 0; h < 2; ++h) {
                    const size_t start = rbw.size();
                    for (int j = 0; j < ph.n_stages; ++j) {
                        const LayerW& lw = layers[ph.st[j].layer];
                        const int ndy = rb_stage_ndy(ph.st[j].kind), ndx = (int)lw.b.size() / ndy;
                        for (int dy = 0; dy < ndy; ++dy)
                            append_resident(rbw, std::vector<std::vector<float>>(lw.b.begin() + ndx * dy, lw.b.begin() + ndx * dy + ndx), lw.n_pad, lw.kk, lw.shift, h);
                    }
                    rbw.resize(start + (size_t)ph.w_bytes / 2, 0);
                }
                phases.push_back(ph);
            }
            for (size_t i = 0; i < phases.size(); ++i) phases[i].w = reinterpret_cast<const unsigned char*>(w_at[i] * 2);   // offsets until the upload below
        }
    }
    const int cells = p->rows * p->cols;
    const int A = p->actions, K = p->policy_channels * cells, VH = p->value_hidden;
    std::vector<float> pfc_wt((size_t)K * A), pfc_b(p->policy_fc_b, p->policy_fc_b + A), vfc1_wt((size_t)cells * VH),
        vfc1_b(p->value_fc1_b, p->value_fc1_b + VH), vfc2_w(p->value_fc2_w, p->value_fc2_w + VH);
    for (int a = 0; a < A; ++a)
        for (int k = 0; k < K; ++k) pfc_wt[(size_t)k * A + a] = p->policy_fc_w[(size_t)a * K + k];
    for (int j = 0; j < VH; ++j)
        for (int k = 0; k < cells; ++k) vfc1_wt[(size_t)k * VH + j] = p->value_fc1_w[(size_t)j * cells + k];
    vfc2_w.push_back(p->value_fc2_b[0]);
    e->upload_bytes = 0;
    constexpr int REPLICAS = 2;
    const size_t one = units.size();
    units.resize(one * REPLICAS);
    for (int r = 1; r < REPLICAS; ++r) std::copy(units.begin(), units.begin() + one, units.begin() + r * one);
    e->dev.wunits_bytes = (long long)(one * sizeof(unsigned short));
    e->dev.replicas = REPLICAS;
    e->dev.nst = MAX_NST;
    while (e->dev.nst > 2 && stream_smem_bytes(C, L, e->dev.nst) > stream_max_smem(C)) e->dev.nst -= 1;
    int rc = e->upload(units, &e->dev.wunits);
    if (!rc) rc = e->upload(head_w, &e->dev.head_w);
    if (!rc && !phases.empty()) {
        rc = e->upload(rbw, &e->rb_weights);
        for (RbPhase& ph : phases) ph.w = reinterpret_cast<const unsigned char*>(e->rb_weights) + reinterpret_cast<size_t>(ph.w);
    }
    if (!rc) e->phases = phases;
    if (!rc) rc = e->upload(bias, &e->dev.bias);
    if (!rc) rc = e->upload(inv_scale, &e->dev.inv_scale);
    if (!rc) rc = e->upload(pfc_wt, &e->dev.pfc_wt);
    if (!rc) rc = e->upload(pfc_b, &e->dev.pfc_b);
    if (!rc) rc = e->upload(vfc1_wt, &e->dev.vfc1_wt);
    if (!rc) rc = e->upload(vfc1_b, &e->dev.vfc1_b);
    if (!rc) rc = e->upload(vfc2_w, &e->dev.vfc2_w);
    std::vector<unsigned long long> flag(2, 0ULL);
    const unsigned long long* fp = e->dev.error_flag;
    if (!rc) rc = e->upload(flag, &fp);
    if (rc) return rc;
    e->dev.error_flag = const_cast<unsigned long long*>(fp);
    e->dev.n_layers = L;
    e->dev.rows = p->rows;
    e->dev.cols = p->cols;
    e->dev.linear = (p->rows > 8 || p->cols > 8) ? 1 : 0;
    e->dev.in_planes = P;
    e->dev.in_ksteps = in_k / KSTEP_CH;
    e->dev.actions = A;
    e->dev.policy_channels = p->policy_channels;
    return SPRL_OK;
}

static int validate(const sprl_network_params* p) {
    if (!p) return fail(SPRL_E_INVALID, "null network parameters");
    if (p->rows < 1 || p->cols < 1 || p->cols > 16 || p->rows * p->cols > TILE_M)
        return fail(SPRL_E_INVALID, "the tcgen05 evaluator tiles boards up to 8x8 (two per MMA) or up to %d cells with rows of at most 16 (one per MMA); got %dx%d", TILE_M, p->rows, p->cols);
    if (p->channels != CH && p->channels != WIDE_CH) return fail(SPRL_E_INVALID, "tower width must be %d or %d channels, got %d", CH, WIDE_CH, p->channels);
    if (p->blocks < 0 || 2 + 2 * p->blocks > MAX_LAYERS) return fail(SPRL_E_INVALID, "unsupported number of residual blocks %d", p->blocks);
    if (p->in_planes < 1 || 3 * p->in_planes > CH) return fail(SPRL_E_INVALID, "unsupported number of input planes %d (at most %d)", p->in_planes, CH / 3);
    if (p->policy_channels < 1 || p->policy_channels > 2 || p->value_channels != 1 || p->value_hidden != p->channels)
        return fail(SPRL_E_INVALID, "unsupported head shape (policy channels %d, value channels %d, value hidden %d; the value hidden layer must be as wide as the tower)",
                    p->policy_channels, p->value_channels, p->value_hidden);
    if (p->actions < 1 || p->actions > HP_STRIDE) return fail(SPRL_E_INVALID, "unsupported action count %d", p->actions);
    int rc = check_conv(p->stem, "stem");
    if (rc) return rc;
    if (p->blocks > 0 && !p->tower) return fail(SPRL_E_INVALID, "null tower");
    for (int i = 0; i < 2 * p->blocks; ++i) { rc = check_conv(p->tower[i], "tower"); if (rc) return rc; }
    if (!p->policy_conv_w || !p->policy_conv_b || !p->policy_fc_w || !p->policy_fc_b || !p->value_conv_w || !p->value_conv_b ||
        !p->value_fc1_w || !p->value_fc1_b || !p->value_fc2_w || !p->value_fc2_b)
        return fail(SPRL_E_INVALID, "null head parameter pointer");
    return SPRL_OK;
}

extern "C" {

int sprl_evalnet_create(int device, const sprl_network_params* params, sprl_evalnet** out) {
    if (!out) return fail(SPRL_E_INVALID, "null output");
    *out = nullptr;
    int rc = validate(params);
    if (rc) return rc;
    rc = use_device(device);
    if (rc) return rc;
    sprl_evalnet* e = new sprl_evalnet();
    memset(&e->dev, 0, sizeof(e->dev));
    e->device = device;
    e->rows = params->rows; e->cols = params->cols; e->in_planes = params->in_planes; e->channels = params->channels;
    e->blocks = params->blocks; e->actions = params->actions; e->policy_channels = params->policy_channels;
    e->value_hidden = params->value_hidden;
    cudaDeviceProp prop;
    cudaError_t err = cudaGetDeviceProperties(&prop, device);
    if (err != cudaSuccess) { delete e; return fail(SPRL_E_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(err)); }
    if (prop.major != 10) { delete e; return fail(SPRL_E_NOGPU, "the tcgen05 evaluator needs an sm_100a device (found sm_%d%d)", prop.major, prop.minor); }
    e->sm_count = prop.multiProcessorCount;
    if (getenv("SPRL_EVALNET_MAX_CTAS")) e->max_ctas = atoi(getenv("SPRL_EVALNET_MAX_CTAS"));
    err = cudaFuncSetAttribute(k_evalnet<false, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, Width<CH>::MAX_SMEM);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(k_evalnet<true, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, Width<CH>::MAX_SMEM);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(k_evalnet<false, WIDE_CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, Width<WIDE_CH>::MAX_SMEM);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(k_evalnet<true, WIDE_CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, Width<WIDE_CH>::MAX_SMEM);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(k_evalnet_resident<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RB_MAX_SMEM);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(k_evalnet_resident<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RB_MAX_SMEM);
    if (err != cudaSuccess) { delete e; return fail(SPRL_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(err)); }
    if (heads_smem_bytes(params->value_hidden, params->policy_channels, params->rows * params->cols) > 227 * 1024) { delete e; return fail(SPRL_E_INVALID, "head layers of %d channels x %d cells do not fit k_heads' shared memory", params->policy_channels, params->rows * params->cols); }
    err = cudaFuncSetAttribute(k_heads<CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);   // the attribute is per process: always the maximum, whatever this evaluator's board
    if (err == cudaSuccess) err = cudaFuncSetAttribute(k_heads<WIDE_CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (err != cudaSuccess) { delete e; return fail(SPRL_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(err)); }
    rc = pack_and_upload(e, params);
    if (rc) { e->release(); delete e; return rc; }
    *out = e;
    return SPRL_OK;
}

int sprl_evalnet_update(sprl_evalnet* e, const sprl_network_params* params) {
    NvtxRange nvtx_range("sprl_evalnet_update");
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    int rc = validate(params);
    if (rc) return rc;
    if (params->rows != e->rows || params->cols != e->cols || params->in_planes != e->in_planes || params->blocks != e->blocks || params->actions != e->actions ||
        params->policy_channels != e->policy_channels || params->channels != e->channels)
        return fail(SPRL_E_INVALID, "sprl_evalnet_update: the network shape changed");
    rc = use_device(e->device);
    if (rc) return rc;
    cudaDeviceSynchronize();
    return pack_and_upload(e, params);
}

int sprl_evalnet_forward(sprl_evalnet* e, const float* d_in, int64_t batch, float* d_logits, float* d_value, void* cuda_stream) {
    return sprl_evalnet_forward_counted(e, d_in, nullptr, batch, d_logits, d_value, cuda_stream);
}

int sprl_evalnet_forward_counted(sprl_evalnet* e, const float* d_in, const uint32_t* d_rows, int64_t batch, float* d_logits,
                                 float* d_value, void* cuda_stream) {
    NvtxRange nvtx_range("sprl_evalnet_forward_counted");
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    if (batch < 0 || (batch > 0 && (!d_in || !d_logits || !d_value))) return fail(SPRL_E_INVALID, "bad argument to sprl_evalnet_forward");
    if (batch == 0) return SPRL_OK;
    cudaError_t err = cudaSetDevice(e->device);
    if (err != cudaSuccess) return fail(SPRL_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(err));
    if (batch > e->head_cap) {
        // grows outside of stream capture only (a captured graph must have seen its batch size before)
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing((cudaStream_t)cuda_stream, &cap);
        if (cap != cudaStreamCaptureStatusNone) return fail(SPRL_E_STATE, "sprl_evalnet_forward: first call with batch %lld inside a stream capture; run one forward of this size before capturing", (long long)batch);
        cudaDeviceSynchronize();
        if (e->head_act) cudaFree(e->head_act);
        e->head_act = nullptr; e->head_cap = 0;
        err = cudaMalloc((void**)&e->head_act, (size_t)batch * (e->policy_channels + 1) * e->rows * e->cols * sizeof(float));
        if (err != cudaSuccess) return fail(SPRL_E_CAPACITY, "cudaMalloc of the head activations failed: %s", cudaGetErrorString(err));
        e->head_cap = batch;
    }
    e->dev.head_act = e->head_act;
    const long long tiles = e->dev.linear ? batch : (batch + 1) / 2;
    const bool resident = !e->phases.empty() && e->path != SPRL_EVALNET_PATH_STREAMING;
    if (e->path == SPRL_EVALNET_PATH_RESIDENT && e->phases.empty())
        return fail(SPRL_E_STATE, "this network does not fit the resident-weight kernel (boards up to 8x8, one stage group per launch within 227 KB)");
    if (e->dev.single_pass && !resident) return fail(SPRL_E_STATE, "the single-pass fp16 mode exists on the resident-weight kernel only");
    if (resident) {
        const long long quads = (tiles + 3) / 4;
        if (e->phases.size() > 1 && quads * 4 > e->act_cap_tiles) {
            cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
            cudaStreamIsCapturing((cudaStream_t)cuda_stream, &cap);
            if (cap != cudaStreamCaptureStatusNone) return fail(SPRL_E_STATE, "sprl_evalnet_forward: first call with batch %lld inside a stream capture; run one forward of this size before capturing", (long long)batch);
            cudaDeviceSynchronize();
            if (e->act) cudaFree(e->act);
            e->act = nullptr; e->act_cap_tiles = 0;
            err = cudaMalloc((void**)&e->act, (size_t)quads * 4 * RB_ACT_TILE_FLOATS * sizeof(float));
            if (err != cudaSuccess) return fail(SPRL_E_CAPACITY, "cudaMalloc of the inter-phase activations failed: %s", cudaGetErrorString(err));
            e->act_cap_tiles = quads * 4;
        }
        int grid = (int)std::min<long long>(2 * quads, (long long)(e->sm_count / 2 * 2));     // one CTA per SM, in pairs
        if (e->max_ctas >= 2) grid = std::min(grid, e->max_ctas / 2 * 2);
        for (RbPhase ph : e->phases) {
            ph.act = e->act;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(grid);
            cfg.blockDim = dim3(RB_THREADS);
            cfg.dynamicSmemBytes = (size_t)rb_smem_bytes(ph, e->dev.linear != 0);
            cfg.stream = (cudaStream_t)cuda_stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            err = e->dev.linear ? cudaLaunchKernelEx(&cfg, k_evalnet_resident<true>, e->dev, ph, d_in, (long long)batch, (const unsigned*)d_rows)
                                : cudaLaunchKernelEx(&cfg, k_evalnet_resident<false>, e->dev, ph, d_in, (long long)batch, (const unsigned*)d_rows);
            e->launches += 1;
            if (err == cudaSuccess) err = cudaGetLastError();
            if (err != cudaSuccess) break;
        }
    } else {
    const bool wide = e->channels == WIDE_CH;
    const int max_grid = e->sm_count * (wide ? Width<WIDE_CH>::CTAS_PER_SM : Width<CH>::CTAS_PER_SM) / CLUSTER * CLUSTER;
    const int grid = (int)std::min<long long>((tiles + CLUSTER - 1) / CLUSTER * CLUSTER, max_grid);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = (size_t)stream_smem_bytes(e->channels, e->dev.n_layers, e->dev.nst);
    cfg.stream = (cudaStream_t)cuda_stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CLUSTER; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    auto* kernel = wide ? (e->dev.linear ? k_evalnet<true, WIDE_CH> : k_evalnet<false, WIDE_CH>)
                        : (e->dev.linear ? k_evalnet<true, CH> : k_evalnet<false, CH>);
    err = cudaLaunchKernelEx(&cfg, kernel, e->dev, d_in, (long long)batch, (const unsigned*)d_rows, d_logits, d_value);
    e->launches += 1;
    if (err == cudaSuccess) err = cudaGetLastError();
    }
    if (err == cudaSuccess) {
        const int hb = e->value_hidden == WIDE_CH ? Heads<WIDE_CH>::HB : Heads<CH>::HB;
        const int hgrid = (int)std::min<long long>((batch + hb - 1) / hb, (long long)e->sm_count);     // one resident CTA per SM (its weights are staged once)
        const size_t hsmem = heads_smem_bytes(e->value_hidden, e->policy_channels, e->rows * e->cols);
        if (e->value_hidden == WIDE_CH)
            k_heads<WIDE_CH><<<hgrid, 256, hsmem, (cudaStream_t)cuda_stream>>>(e->dev, (long long)batch, (const unsigned*)d_rows, d_logits, d_value);
        else
            k_heads<CH><<<hgrid, 256, hsmem, (cudaStream_t)cuda_stream>>>(e->dev, (long long)batch, (const unsigned*)d_rows, d_logits, d_value);
        e->launches += 1;
        err = cudaGetLastError();
    }
    if (err != cudaSuccess) return fail(SPRL_E_CUDA, "k_evalnet launch failed: %s", cudaGetErrorString(err));
    return SPRL_OK;
}

int sprl_evalnet_status(sprl_evalnet* e, uint64_t* launches) {
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    cudaError_t err = cudaSetDevice(e->device);
    if (err != cudaSuccess) return fail(SPRL_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(err));
    unsigned long long flag[2] = { 0, 0 };
    err = cudaMemcpy(flag, e->dev.error_flag, sizeof(flag), cudaMemcpyDeviceToHost);
    if (err != cudaSuccess) return fail(SPRL_E_CUDA, "evaluator kernel failed: %s", cudaGetErrorString(err));
    if (flag[0]) return fail(SPRL_E_CUDA, "evaluator kernel timed out on a pipeline barrier (code %llx)", flag[0]);
    if (flag[1]) return fail(SPRL_E_STATE, "an input or activation exceeded %.0f, the range of the fp16-split evaluator; its outputs were clamped", HALF_MAX / ACT_SCALE);
    if (launches) *launches = e->launches;
    return SPRL_OK;
}

int sprl_evalnet_info(sprl_evalnet* e, int64_t* upload_bytes, int32_t* ring_stages, int32_t* smem_bytes) {
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    if (upload_bytes) *upload_bytes = e->upload_bytes;
    if (ring_stages) *ring_stages = e->dev.nst;
    if (smem_bytes) {
        *smem_bytes = stream_smem_bytes(e->channels, e->dev.n_layers, e->dev.nst);
        if (!e->phases.empty() && e->path != SPRL_EVALNET_PATH_STREAMING) {      // the resident kernel: its largest phase
            *smem_bytes = 0;
            for (const RbPhase& ph : e->phases) *smem_bytes = std::max(*smem_bytes, rb_smem_bytes(ph, e->dev.linear != 0));
        }
    }
    return SPRL_OK;
}

int sprl_evalnet_set_path(sprl_evalnet* e, int path) {
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    if (path < SPRL_EVALNET_PATH_AUTO || path > SPRL_EVALNET_PATH_RESIDENT) return fail(SPRL_E_INVALID, "unknown evaluator path %d", path);
    if (path == SPRL_EVALNET_PATH_RESIDENT && e->phases.empty())
        return fail(SPRL_E_STATE, "this network does not fit the resident-weight kernel");
    e->path = path;
    return SPRL_OK;
}

int sprl_evalnet_set_precision(sprl_evalnet* e, int precision) {
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    if (precision != SPRL_EVALNET_PRECISION_FP32_SPLIT && precision != SPRL_EVALNET_PRECISION_FP16) return fail(SPRL_E_INVALID, "unknown evaluator precision %d", precision);
    if (precision == SPRL_EVALNET_PRECISION_FP16 && (e->phases.empty() || e->path == SPRL_EVALNET_PATH_STREAMING))
        return fail(SPRL_E_STATE, "the single-pass fp16 mode exists on the resident-weight kernel only");
    e->dev.single_pass = precision == SPRL_EVALNET_PRECISION_FP16 ? 1 : 0;
    return SPRL_OK;
}

int sprl_evalnet_phases(sprl_evalnet* e) {
    if (!e) return fail(SPRL_E_INVALID, "null evaluator");
    return (e->phases.empty() || e->path == SPRL_EVALNET_PATH_STREAMING) ? 0 : (int)e->phases.size();
}

void sprl_evalnet_destroy(sprl_evalnet* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    e->release();
    delete e;
}

}  // extern "C"
