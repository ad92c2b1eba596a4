// absorb_head_tc.cu — the absorbing-rate transformer head on tcgen05 tensor cores (sm_100a).
//
// AbsorbingGenerator.absorbing_head (mp/models/generative/absorbing/absorbing_flows.py:94-131):
// Linear(H+2 -> 128) on [last local hidden, one_hot(mask)], then n_blocks x (ResnetBlock, AttnBlock)
// (mp/models/architectures/gsdm.py:38-66,142-168) over the N particle slots of a jet, then
// Linear(128->128), Linear(128->1).  72 MFLOP per jet-step (SURVEY.md §8d): ~99 % of the absorbing
// flow's arithmetic, and real GEMM work (M = 128 particles, N = K = 128 channels).
//
// One CTA (256 threads) owns one jet at a time (persistent over jets).  Particle r = TMEM lane r is served by two
// threads: warp w < 4 handles channels [0,64) of rows 32w..32w+31, warp w+4 channels [64,128) of the same rows —
// which is also "one thread per (query, attention head)", so softmax rows and their 1/rowsum never leave a thread.
//   * the residual stream X [128 x 128] fp32 lives in TMEM for the whole head; conv2 and proj_out
//     accumulate straight into it (the residual add is the accumulate flag), their biases ride on
//     one more K-step against a ones tile;
//   * every 1x1 conv is 8 tcgen05.mma M128 x N128 x K16 (bf16 operands, canonical no-swizzle
//     K-major tiles); weights stream L2 -> shared memory with cp.async.bulk (1-D TMA) into a
//     two-stage ring, one 36 KB slot per matrix, one phase ahead of their use;
//   * attention per head: S = Q K^T (4 K-steps) into TMEM, row softmax by the thread that owns the
//     query (its lane holds the whole row — no cross-thread reduction), P as bf16 A operand,
//     O = P V with V consumed as an MN-major B operand (no transpose), 1/rowsum applied to O;
//   * GroupNorm(32) statistics: per-thread partial sums over its 128 channels, one shared-memory
//     reduction across particles, then normalise + swish while packing the next A operand.
// Numerics: bf16 operands, fp32 accumulate / statistics / softmax.  Checked against the fp32 oracle
// with the tolerance stated in tests/test_gpu_absorbing.py.
//
// Round 2 — dead slots once, several jets per tile.  The reference runs the stack over ALL N slots of a jet, padded ones
// included (no attention mask, GroupNorm statistics over every slot).  The stack is permutation-equivariant and every padded slot
// carries the same input row, so all padded slots of a jet hold the SAME row at every depth: the kernel computes one
// representative dead row per jet and gives it the weight n_dead wherever rows are summed — GroupNorm sums, softmax
// denominators and P V (the weight multiplies the key's column of P), the slot mean of the per-jet heads — which is exact.  A jet
// then needs m_live + 1 rows, rounded up to 32-row quarters of the 128-row tile (= one warp per channel slice, so the statistics
// of a jet are sums over whole warps and the softmax masks whole 32-key chunks); a pre-pass bins the jets by quarters needed
// (after checking that their padded slots really are identical — otherwise the jet keeps a tile of its own with one row per
// slot) and the kernel walks tiles composed [4] | [3,1] | [2,2] | [2,1,1] | [1,1,1,1] with block-diagonal attention.  At
// JetClass-like multiplicities (mean 45 of 128) a tile carries 2.1 jets; in the trans-dimensional sampler, where jets grow from
// one particle, four.
#include <cuda_bf16.h>

#include <vector>

#include "mmb_device.cuh"
#include "mmb_internal.h"
#include "tcgen05.cuh"

namespace mmb {
namespace {

constexpr int kC = 128;            // transformer width this kernel is built for
constexpr int kHeads = 2;            // 64 channels per head
constexpr int kMaxBlocks = 4;

// fp32 side table (floats), per block then the per-particle output vector
struct HeadTable {
    // per block: n1g n1b b1 n2g n2b n3g n3b  (7 x 128); the q / k / v biases live in the operand image or are folded away
    static constexpr int kPerBlock = 7 * kC;
    __host__ __device__ static int rate_w(int nblk) { return nblk * kPerBlock; }       // [128] per-particle output vector
    __host__ __device__ static int rate_c(int nblk) { return nblk * kPerBlock + kC; }  // its constant
    __host__ __device__ static int floats(int nblk) { return nblk * kPerBlock + kC + 4; }
};

struct HeadParams {
    const uint8_t* image;    // n_seq slots of kSlot bytes (bf16 operand tiles)
    const float* table;      // HeadTable
    int n_blocks, H;
    int mode, S;             // TfStackIO::mode; one-hot width (modes 1, 2)
    const float* hidden;     // [B,N,H]
    const uint8_t* mask;     // [B,N]
    const float* onehot;     // [B,N,S]   (modes 1, 2)
    const float* x;          // [B,N,3]   (mode 2)
    const int32_t* nearest;  // [B]       (mode 2)
    const float* tbias;      // [B or 1][n_blocks][128]
    int tbias_stride;
    int B, N;
    float* logit_out;        // [B,N] per-particle output
    int n_jet;               // > 0: also write the mean of X over the N slots
    float* jet_out;          // [B][128] slot means (the per-jet head consumes them)
    const int32_t* pack;     // PackScratch of this call (tf_pack_kernel), or null: one jet per tile, one row per slot
};

// ---- packing pre-pass ---------------------------------------------------------------------------------------------------------
// scratch (int32): counts[8] (jets needing q quarters at [q], q = 1..4; [5] = tiles) | info[B] (live count | packable << 16) |
// lists[4][B] | tile records [<= B][kTileRec]
constexpr int kMaxSeg = 4;
constexpr int kTileRec = 24;   // n_seg, jet[4], q0[4], nq[4], m[4], packed[4] (+ padding): the head of TileState
struct PackScratch {
    __host__ __device__ static size_t ints(int B) { return 8 + (size_t)B * 5 + (size_t)B * kTileRec; }
    __host__ __device__ static const int32_t* list(const int32_t* p, int B, int q) { return p + 8 + (size_t)B * q; }   // q = 1..4
    __host__ __device__ static const int32_t* tiles(const int32_t* p, int B) { return p + 8 + (size_t)B * 5; }
};

// tile t of a call -> its jets.  Tiles: [4] x n4 | [3 (+1)] x n3 | [2,2] x n2/2 | [2 (+1) (+1)] if n2 is odd | [1,1,1,1] ...
struct TileDesc {
    int n_seg, jet[kMaxSeg], q0[kMaxSeg], nq[kMaxSeg];
};
__device__ inline int pack_tiles(const int32_t* pack) {
    const int n1 = pack[1], n2 = pack[2], n3 = pack[3], n4 = pack[4];
    const int a = min(n3, n1), b = (n2 & 1) ? min(2, n1 - a) : 0;
    return n4 + n3 + n2 / 2 + (n2 & 1) + (n1 - a - b + 3) / 4;
}
__device__ inline void tile_desc(const int32_t* pack, int B, int t, TileDesc& d) {
    const int n1 = pack[1], n2 = pack[2], n3 = pack[3], n4 = pack[4];
    const int32_t *l1 = PackScratch::list(pack, B, 1), *l2 = PackScratch::list(pack, B, 2), *l3 = PackScratch::list(pack, B, 3),
                  *l4 = PackScratch::list(pack, B, 4);
    const int a = min(n3, n1), b = (n2 & 1) ? min(2, n1 - a) : 0;
    d.n_seg = 0;
    auto add = [&](int jet, int nq) {
        d.q0[d.n_seg] = d.n_seg ? d.q0[d.n_seg - 1] + d.nq[d.n_seg - 1] : 0;
        d.jet[d.n_seg] = jet; d.nq[d.n_seg] = nq; ++d.n_seg;
    };
    if (t < n4) { add(l4[t], 4); return; }
    t -= n4;
    if (t < n3) { add(l3[t], 3); if (t < a) add(l1[t], 1); return; }
    t -= n3;
    if (t < n2 / 2) { add(l2[2 * t], 2); add(l2[2 * t + 1], 2); return; }
    t -= n2 / 2;
    if (n2 & 1) {
        if (t == 0) { add(l2[n2 - 1], 2); for (int i = 0; i < b; ++i) add(l1[a + i], 1); return; }
        t -= 1;
    }
    for (int i = 0; i < 4; ++i) {
        const int idx = a + b + 4 * t + i;
        if (idx < n1) add(l1[idx], 1);
    }
}

// tile t's jets written out as a record the main kernel fetches with one coalesced load
__device__ inline void tile_record(int32_t* __restrict__ pack, int B, int t) {
    TileDesc d;
    tile_desc(pack, B, t, d);
    int32_t* rec = pack + 8 + (size_t)B * 5 + (size_t)t * kTileRec;
    rec[0] = d.n_seg;
    for (int sg = 0; sg < kMaxSeg; ++sg) {
        const bool on = sg < d.n_seg;
        const int info = on ? pack[8 + d.jet[sg]] : 0;
        rec[1 + sg] = on ? d.jet[sg] : 0; rec[5 + sg] = on ? d.q0[sg] : 0; rec[9 + sg] = on ? d.nq[sg] : 0;
        rec[13 + sg] = info & 0xffff; rec[17 + sg] = info >> 16;
    }
}

// warp per jet: live count, are the inputs of all padded slots bit-identical (mode 0: hidden; mode 1: hidden + onehot; mode 2:
// masked, always), quarters needed; appended to the list of its class (order irrelevant: a jet's rows only ever meet its own)
__global__ void __launch_bounds__(256) tf_pack_kernel(const uint8_t* __restrict__ mask, const float* __restrict__ hidden, int H,
                                                      const float* __restrict__ onehot, int S, int mode, int B, int N, int32_t* __restrict__ pack) {
    const int jet = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (jet >= B) return;
    int m = 0, first_dead = N;
    for (int n0 = 0; n0 < N; n0 += 32) {
        const int n = n0 + lane;
        const unsigned live = __ballot_sync(0xffffffffu, n < N && mask[(size_t)jet * N + n] != 0);
        const unsigned dead = ~live & (N - n0 >= 32 ? 0xffffffffu : ((1u << (N - n0)) - 1u));
        m += __popc(live);
        if (first_dead == N && dead) first_dead = n0 + __ffs(dead) - 1;
    }
    bool same = true;
    if (mode != 2 && first_dead < N) {   // value comparison: -0.0 == +0.0 (x * mask leaves either), NaN never equals
        const float* h0 = hidden + ((size_t)jet * N + first_dead) * H;
        const float* o0 = mode == 1 ? onehot + ((size_t)jet * N + first_dead) * S : nullptr;
        for (int n = first_dead + 1 + lane; n < N; n += 32) {
            if (mask[(size_t)jet * N + n]) continue;
            const float* h = hidden + ((size_t)jet * N + n) * H;
            for (int i = 0; i < H; ++i) same = same && h[i] == h0[i];
            if (o0) {
                const float* o = onehot + ((size_t)jet * N + n) * S;
                for (int i = 0; i < S; ++i) same = same && o[i] == o0[i];
            }
        }
    }
    same = __all_sync(0xffffffffu, same);
    if (lane == 0) {
        const int rows = same ? m + (m < N ? 1 : 0) : N;         // not packable: one row per slot
        const int q = (rows + 31) / 32;
        pack[8 + jet] = m | ((same ? 1 : 0) << 16);
        const int pos = atomicAdd(pack + q, 1);
        pack[8 + (size_t)B * q + pos] = jet;
    }
}

// one thread per tile (a separate launch: folded into the last block of tf_pack_kernel it ran serially, 20 us slower at 4096 jets)
__global__ void __launch_bounds__(256) tf_tiles_kernel(int32_t* __restrict__ pack, int B) {
    const int n_tiles = pack_tiles(pack);
    if (blockIdx.x == 0 && threadIdx.x == 0) pack[5] = n_tiles;
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t < n_tiles) tile_record(pack, B, t);
}

constexpr int kSmemW = 2 * kSlot;                         // weight ring
constexpr int kOffA = kSmemW, kOffQ = kOffA + 32768, kOffK = kOffQ + 32768, kOffV = kOffK + 32768;
constexpr int kOffOnes = kOffV + 32768, kOffTab = kOffOnes + 4096;

constexpr int kCW = 32;                   // accumulator columns per thread (16 = 32 warps: measured slower, 393 vs 435 TFLOP/s)
constexpr int kNQ = kC / kCW;             // channel slices per row
constexpr int kThreads = 128 * kNQ;       // 16 warps at kCW = 32

__device__ __forceinline__ float tanh_fast(float a) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(a));
    return t;
}

// One CTA owns one TILE at a time: 128 rows = up to four jets in 32-row quarters (see the header).  Thread (r, cq): row r = TMEM
// lane r (warp & 3 selects the lane quarter the warp may touch), channel slice cq = warp >> 2 -> kCW consecutive accumulator
// columns = one tcgen05.ld per pass.
__global__ void __launch_bounds__(kThreads, 1) absorb_head_tc_kernel(const HeadParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr int CW = kCW, NQ = kNQ, G = CW / 4, HQ = NQ / 2;   // HQ: threads per (row, attention head)
    static_assert(CW == 32, "a softmax key chunk must be one 32-row quarter of the tile");
    __shared__ uint32_t s_tmem_slot;
    __shared__ __align__(8) uint64_t s_bars[4];             // full[0], full[1], mma, mma2 (the v GEMM that runs under the softmax)
    __shared__ __align__(16) float s_part[4 * NQ][CW];      // per-warp partial sums (GroupNorm statistics / column sums)
    // GroupNorm scale / shift per (segment, channel) and the softmax row max / row sum per (channel slice, row) are never alive
    // at the same time: one buffer
    __shared__ __align__(16) float s_shared[kMaxSeg * 256];
    float (*s_stat)[256] = reinterpret_cast<float (*)[256]>(s_shared);            // [segment][scale 128 | shift 128]
    float (*s_rowx)[128] = reinterpret_cast<float (*)[128]>(s_shared);            // [NQ][128]
    float (*s_sum)[128] = reinterpret_cast<float (*)[128]>(s_shared + NQ * 128);  // [NQ][128]
    float (*s_dot)[128] = s_rowx;                           // per-row output partials (after the last softmax)
    // The jets of a tile, the row -> slot map and the row weights; double-buffered: the next tile's state is prepared, step by
    // step, while the current tile computes (descriptor -> masks -> row map -> cp.async of the rows' inputs), so that no global
    // load latency sits between two tiles.
    struct TileState {
        int n_seg, seg_jet[kMaxSeg], seg_q0[kMaxSeg], seg_nq[kMaxSeg], seg_m[kMaxSeg], seg_packed[kMaxSeg];   // = a tile record
        int qseg[4];                 // row quarter -> segment, -1: empty
        int qwt[4];                  // row quarter holds a row of weight != 1 (softmax then applies lw / kb to its keys)
        int seg_near[kMaxSeg];       // mode 2: the jet's nearest particle
        uint32_t mbits[kMaxSeg][4];  // live mask of each jet, one bit per slot
        int slot[128];               // row -> slot of its jet (-1: unused row)
        alignas(16) float w[128];    // row weight: 1 live, n_dead for a jet's representative padded row, 0 unused
        alignas(16) float lw[128];   // log2(w): added to a key's exponent, P = w * exp(.); -inf for unused rows
        alignas(16) float kb[128];   // 0 / -3e38: added to a key's score in the row-max pass
    };
    __shared__ TileState s_tile[2];
    TileState *ts = &s_tile[0], *tn = &s_tile[1];
    // the warp index is broadcast so that the compiler sees it (and what derives from it) as warp-uniform
    const int tid = threadIdx.x, r = tid & 127, cq = tid >> 7, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int qq = warp & 3;                                // this warp's row quarter
    const int nblk = p.n_blocks, n_seq = 1 + 6 * nblk;
    uint8_t *sA = smem + kOffA, *sQ = smem + kOffQ, *sK = smem + kOffK, *sV = smem + kOffV, *sOnes = smem + kOffOnes;
    float* sTab = reinterpret_cast<float*>(smem + kOffTab);
    float* s_bias2 = sTab + HeadTable::floats(nblk);        // [segment][nblk][128] conv1 bias + the jet's time term
    uint8_t* sA0 = sV;                                      // [128 x 32] proj_in operand, aliases V (dead at tile start)

    for (int i = tid; i < HeadTable::floats(nblk); i += kThreads) sTab[i] = __ldg(p.table + i);
    for (int i = tid; i < 256; i += kThreads) reinterpret_cast<uint4*>(sOnes)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    const uint32_t bar_full0 = smem_u32(&s_bars[0]), bar_full1 = smem_u32(&s_bars[1]), bar_mma = smem_u32(&s_bars[2]), bar_mma2 = smem_u32(&s_bars[3]);
    if (tid == 0) { mbar_init(bar_full0, 1); mbar_init(bar_full1, 1); mbar_init(bar_mma, 1); mbar_init(bar_mma2, 1); }
    if (warp == 0) tmem_alloc(smem_u32(&s_tmem_slot), 512);
    fence_barrier_init();
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, s_tmem_slot, 0);   // broadcast: provably warp-uniform, so UMMA operands stay in uniform registers
    const uint32_t lane_off = ((uint32_t)(qq * 32) << 16);           // this warp's TMEM lane quarter
    const int col0 = cq * CW;                                        // this thread's accumulator columns
    const uint32_t dX = tmem, dACC = tmem + 128, dS0 = tmem + 256, dS1 = tmem + 384;

    const int n_tiles = p.pack ? p.pack[5] : p.B;
    const int32_t* tile_recs = p.pack ? PackScratch::tiles(p.pack, p.B) : nullptr;
    const int my_tiles = n_tiles > (int)blockIdx.x ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const uint32_t total_mats = (uint32_t)my_tiles * n_seq;
    const uint32_t wbase = smem_u32(smem);
    // Ring slot 0 = [bias tile | weight tile], slot 1 = [weight tile | bias tile]: the two weight tiles are adjacent in shared
    // memory, so a pair of streamed matrices can be consumed as ONE [256 x 128] B operand (the fused q/k GEMM).
    auto w_addr = [&](uint32_t slot) { return wbase + (slot ? kSlot : kSlot - kSlotBias); };
    auto b_addr = [&](uint32_t slot) { return wbase + (slot ? kSlot + kSlotBias : 0u); };
    auto issue_load = [&](uint32_t i) {  // thread 0 only
        const uint32_t bar = (i & 1) ? bar_full1 : bar_full0;
        const uint8_t* src = p.image + (size_t)(i % n_seq) * kSlot;
        mbar_expect_tx(bar, kSlot);
        bulk_g2s(w_addr(i & 1), src, kSlotBias, bar);
        bulk_g2s(b_addr(i & 1), src + kSlotBias, kSlot - kSlotBias, bar);
    };
    if (tid == 0) {
        if (total_mats > 0) issue_load(0);
        if (total_mats > 1) issue_load(1);
    }
    uint32_t wseq = 0, mma_phase = 0, mma2_phase = 0;
    constexpr uint32_t idesc128 = instr_desc(128, 128, false), idesc64mn = instr_desc(128, 64, true), idesc256 = instr_desc(128, 256, false);
    const uint64_t ones_desc = smem_desc(smem_u32(sOnes), 128, 256);
    const uint32_t aA = smem_u32(sA), aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV);

    // D (+)= A[128 x 16*nk] * W^T with the streamed matrix `wseq`; optional bias K-step; commit.  Thread 0.
    // MMA issue: warp 0 enters as a whole, broadcasts the streamed-matrix counter (a tcgen05.mma whose descriptor operands are
    // not provably warp-uniform is wrapped by the compiler in an elect/broadcast loop of ~15 instructions per instruction), and
    // one elected lane issues.
    auto mma_issue = [&](auto&& fn) {
        if (warp == 0) {
            const uint32_t ws = __shfl_sync(0xffffffffu, wseq, 0);
            if (elect_one()) fn(ws);
        }
    };
    auto gemm_w = [&](uint32_t wseq, uint32_t d, uint32_t a_addr, uint32_t a_sbo, int nk, bool accumulate, bool bias, uint32_t bar_done) {
        const uint32_t wb = w_addr(wseq & 1);
        mbar_wait((wseq & 1) ? bar_full1 : bar_full0, (wseq >> 1) & 1);
        tc_fence_after();
        // descriptors advance by 256 B per K-step: +16 in the (address >> 4) field, no per-step re-encoding
        const uint64_t ad = smem_desc(a_addr, 128, a_sbo), wd = smem_desc(wb, 128, 2048);
#pragma unroll 8
        for (int j = 0; j < nk; ++j) umma(d, ad + (uint64_t)(j * 16), wd + (uint64_t)(j * 16), idesc128, (accumulate || j > 0) ? 1u : 0u);
        if (bias) umma(d, ones_desc, smem_desc(b_addr(wseq & 1), 128, 256), idesc128, 1u);
        umma_commit(bar_done);
    };
    // The q and k projections as one M128 x N256 GEMM over the two ring slots: D columns [0,128) come from the matrix in
    // slot 0, [128,256) from the one in slot 1 (which of q, k sits where alternates from tile to tile: n_seq is odd).
    // The q bias rides on one more K-step into q's half.  Thread 0.
    auto gemm_qk = [&](uint32_t wseq, uint32_t d, uint32_t a_addr) {
        mbar_wait((wseq & 1) ? bar_full1 : bar_full0, (wseq >> 1) & 1);
        mbar_wait(((wseq + 1) & 1) ? bar_full1 : bar_full0, ((wseq + 1) >> 1) & 1);
        tc_fence_after();
        const uint64_t ad = smem_desc(a_addr, 128, 2048), wd = smem_desc(w_addr(0), 128, 2048);
#pragma unroll
        for (int j = 0; j < 8; ++j) umma(d, ad + (uint64_t)(j * 16), wd + (uint64_t)(j * 16), idesc256, j > 0 ? 1u : 0u);
        umma(d + (wseq & 1) * 128, ones_desc, smem_desc(b_addr(wseq & 1), 128, 256), idesc128, 1u);
        umma_commit(bar_mma);
    };
    // all threads: wait for the committed MMAs; the ring slots of the consumed matrices are free again -> prefetch
    auto mma_done = [&](int used_weights) {
        mbar_wait(bar_mma, mma_phase); mma_phase ^= 1;
        tc_fence_after();
        for (int i = 0; i < used_weights; ++i) {
            if (tid == 0 && wseq + 2 < total_mats) issue_load(wseq + 2);
            ++wseq;
        }
    };

    // per-tile facts of this thread (set at the head of every tile)
    int seg = 0;             // segment (jet) of this warp's quarter, -1: the quarter is empty; warp-uniform
    int seg_first = 0;       // first quarter of that segment
    int seg_nq = 4;          // its quarters
    float w_row = 1.0f;      // weight of row r
    const float inv_slots = 1.0f / (4.0f * (float)p.N);

    // GroupNorm(32 groups of 4 channels) over the N slots of each jet of the tile (+ per-channel bias) -> bf16 A tile.  A jet's
    // statistics are weighted sums over the rows of its quarters.  One TMEM read: the values stay in registers across the
    // statistics exchange, which only involves the four warps of a channel slice (named barrier 1 + cq, 128 threads).
    auto group_norm_to_A = [&](uint32_t d_src, const float* bias /*nullable, smem, per segment*/, const float* gamma, const float* beta,
                               bool swish) {
        float v[CW];
        tmem_ld32(d_src + lane_off + col0, v);
        if (bias) {
#pragma unroll
            for (int j = 0; j < CW; j += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(bias + col0 + j);
                fadd2(v[j], v[j + 1], v[j], v[j + 1], b4.x, b4.y);
                fadd2(v[j + 2], v[j + 3], v[j + 2], v[j + 3], b4.z, b4.w);
            }
        }
        float st[2 * G];   // G group sums, G group sums of squares
        const bool counts = w_row > 0.0f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
            float s0, s1, q0, q1;
            fadd2(s0, s1, v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
            fmul2(q0, q1, v[4 * g], v[4 * g + 1], v[4 * g], v[4 * g + 1]);
            ffma2(q0, q1, v[4 * g + 2], v[4 * g + 3], v[4 * g + 2], v[4 * g + 3], q0, q1);
            st[g] = counts ? w_row * (s0 + s1) : 0.0f;        // select, not multiply: unused rows may hold anything
            st[G + g] = counts ? w_row * (q0 + q1) : 0.0f;
        }
        warp_halving_sum<2 * G>(st, lane);
        if ((lane & (32 / (2 * G) - 1)) == 0) s_part[warp][warp_halving_index<2 * G>(lane)] = st[0];
        named_bar(1 + cq, 128);
        if (seg >= 0 && qq == seg_first && lane < CW) {  // first warp of the jet in this slice, one lane per channel: y = x*scale + shift
            const int c = col0 + lane, gi = lane >> 2, w0 = cq * 4 + seg_first;
            float sp[4], qp[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {   // the jet's quarters (independent loads), added in a fixed order
                const bool on = i < seg_nq;
                sp[i] = on ? s_part[w0 + i][gi] : 0.0f;
                qp[i] = on ? s_part[w0 + i][G + gi] : 0.0f;
            }
            const float s = (sp[0] + sp[1]) + (sp[2] + sp[3]), q = (qp[0] + qp[1]) + (qp[2] + qp[3]);
            const float mean = s * inv_slots;
            const float var = fmaxf(q * inv_slots - mean * mean, 0.0f);
            const float h = swish ? 0.5f : 1.0f;   // swish(a) = a/2 * tanh(a/2) + a/2: the halving rides on the affine
            const float scale = rsqrtf(var + 1e-6f) * gamma[c] * h;
            s_stat[seg][c] = scale;
            s_stat[seg][128 + c] = fmaf(-mean, scale, beta[c] * h);
        }
        named_bar(1 + cq, 128);
        const float* stat = s_stat[seg < 0 ? 0 : seg];
#pragma unroll
        for (int j = 0; j < CW; j += 4) {
            const float4 sc = *reinterpret_cast<const float4*>(stat + col0 + j);
            const float4 sh = *reinterpret_cast<const float4*>(stat + 128 + col0 + j);
            ffma2(v[j], v[j + 1], v[j], v[j + 1], sc.x, sc.y, sh.x, sh.y);
            ffma2(v[j + 2], v[j + 3], v[j + 2], v[j + 3], sc.z, sc.w, sh.z, sh.w);
        }
        if (swish) {
#pragma unroll
            for (int j = 0; j < CW; j += 2) {
                const float t0 = tanh_fast(v[j]), t1 = tanh_fast(v[j + 1]);
                ffma2(v[j], v[j + 1], v[j], v[j + 1], t0, t1, v[j], v[j + 1]);
            }
        }
        if (seg < 0) {   // empty quarter: keep the operand rows finite (they meet nobody, but NaN x 0 would)
#pragma unroll
            for (int j = 0; j < CW; ++j) v[j] = 0.0f;
        }
        store_row<CW>(sA, r, col0, v);
        tc_fence_before();
        fence_proxy_async();
        __syncthreads();
    };
    // q / k / v biases are handled algebraically: q rides on an extra K-step; k is a per-query constant in the logits
    // (softmax-invariant) and is dropped; v is folded into the proj_out bias because softmax rows sum to one.
    // ---- preparation of a tile, in four steps that are spread over the phases of the previous tile -------------------------------
    float* sStage = reinterpret_cast<float*>(sV + 16384);    // [128 rows][32 floats]: hidden | onehot | x | x of the nearest particle
    float* sTbias = reinterpret_cast<float*>(sV + 8192);     // [segment][nblk][128] raw time terms (the proj_in operand sits below)
    int desc_reg = 0;
    uint32_t mask_reg = 0;
    int near_reg = 0;
    // Warps 8..15 do the preparation: warp 0 issues the GEMMs and must never sit on a global load.
    const int pw = warp - 8;
    // 1. the tile's record -> one register of lanes 0..20 of warp 8 (a load in flight, nothing waits for it)
    auto desc_issue = [&](int tile) {
        if (pw == 0 && lane < 21) {
            if (tile_recs) desc_reg = __ldg(tile_recs + (size_t)tile * kTileRec + lane);
            else desc_reg = lane == 0 ? 1 : lane == 1 ? tile : lane == 9 ? (p.N + 31) / 32 : 0;   // one jet per tile, one row per slot
        }
    };
    // 2. record -> shared memory (warp 8), quarter -> segment table
    auto desc_commit = [&](TileState* t) {
        if (pw == 0) {
            if (lane < 21) reinterpret_cast<int*>(t)[lane] = desc_reg;
            __syncwarp();
            if (lane < 4) {
                int sgq = -1;
                for (int sg = 0; sg < t->n_seg; ++sg)
                    if (lane >= t->seg_q0[sg] && lane < t->seg_q0[sg] + t->seg_nq[sg]) sgq = sg;
                t->qseg[lane] = sgq;
            }
        }
    };
    // 3. warp 8 + sg: the mask bytes of jet sg (and its nearest particle) -> registers
    auto masks_issue = [&](const TileState* t) {
        if (pw >= 0 && pw < t->n_seg) {
            const int jet = t->seg_jet[pw];
            mask_reg = 0;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const int n = 32 * w + lane;
                if (n < p.N) mask_reg |= (uint32_t)(p.mask[(size_t)jet * p.N + n] != 0) << (8 * w);
            }
            near_reg = p.mode == 2 ? __ldg(p.nearest + jet) : 0;
        }
    };
    // 4. warp 8 + sg: mask bits of jet sg, then slot and weight of each of its rows (live slots scatter themselves to the row of
    // their rank; the row after the last live one represents the padded slots)
    auto rowmap_build = [&](TileState* t) {
        auto set_row = [&](int row, int slot, float w) {
            t->slot[row] = slot;
            t->w[row] = w;
            t->lw[row] = w > 0.0f ? __log2f(w) : -INFINITY;
            t->kb[row] = w > 0.0f ? 0.0f : -3.0e38f;
        };
        if (pw >= 0 && pw < t->n_seg) {
            const int sg = pw, m = t->seg_m[sg], packed = t->seg_packed[sg], base = 32 * t->seg_q0[sg];
            uint32_t bits[4];
#pragma unroll
            for (int w = 0; w < 4; ++w) bits[w] = __ballot_sync(0xffffffffu, (mask_reg >> (8 * w)) & 1u);
            if (lane < 4) t->mbits[sg][lane] = lane == 0 ? bits[0] : lane == 1 ? bits[1] : lane == 2 ? bits[2] : bits[3];
            if (lane == 0) t->seg_near[sg] = near_reg;
            for (int q = 0; q < t->seg_nq[sg]; ++q) {
                const int i = 32 * q + lane;
                if (!packed && i < p.N) set_row(base + i, i, 1.0f);     // one row per slot, live or not
                else set_row(base + i, -1, 0.0f);
            }
            if (lane < t->seg_nq[sg])   // all rows of weight 1: one per slot with N a multiple of 32, or a packed quarter full of live slots
                t->qwt[t->seg_q0[sg] + lane] = packed ? (m < 32 * (lane + 1)) : (p.N < 32 * (lane + 1));
            __syncwarp();
            if (packed) {
                int before = 0, first_dead = -1;
#pragma unroll
                for (int wd = 0; wd < 4; ++wd) {
                    const int n = 32 * wd + lane;
                    if ((bits[wd] >> lane) & 1u) set_row(base + before + __popc(bits[wd] & ((1u << lane) - 1u)), n, 1.0f);
                    before += __popc(bits[wd]);
                    const uint32_t dead = ~bits[wd] & (p.N - 32 * wd >= 32 ? 0xffffffffu : (p.N > 32 * wd ? (1u << (p.N - 32 * wd)) - 1u : 0u));
                    if (first_dead < 0 && dead) first_dead = 32 * wd + __ffs(dead) - 1;
                }
                if (lane == 0 && m < p.N) set_row(base + m, first_dead, (float)(p.N - m));   // the p.N - m identical padded slots
            }
        }
        if (pw >= 4) {   // rows of empty quarters
            const int q = pw - 4;
            if (t->qseg[q] < 0) set_row(32 * q + lane, -1, 0.0f);
        }
    };
    // 5. gather the inputs of the tile's rows (and the time terms of its jets) into the staging area with cp.async; the V tile
    // they alias is dead once the last P V GEMM of a tile has completed
    auto cp4 = [&](float* dst, const float* src) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
    };
    auto cp16 = [&](float* dst, const float* src) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
    };
    // staging row r: float i sits at 16-byte chunk (i / 4) ^ (r & 7), so that the eight chunks a quarter-warp reads (same
    // chunk number, consecutive rows) fall in different banks
    auto stage_at = [&](int row, int i) { return sStage + row * 32 + ((((i >> 2) ^ (row & 7)) << 2) | (i & 3)); };
    auto rows_prefetch = [&](const TileState* t) {
        const int sgq = t->qseg[qq], slot = t->slot[r];
        if (sgq >= 0 && slot >= 0) {
            const int jet = t->seg_jet[sgq];
            const size_t pi = (size_t)jet * p.N + slot;
            if (cq == 0) {
                const float* src = p.hidden + pi * p.H;
                if (((p.H & 3) | (int)(reinterpret_cast<uintptr_t>(p.hidden) & 15)) == 0) for (int i = 0; i < p.H; i += 4) cp16(stage_at(r, i), src + i);
                else for (int i = 0; i < p.H; ++i) cp4(stage_at(r, i), src + i);
            } else if (cq == 1 && p.mode) {
                const float* src = p.onehot + pi * p.S;
                if (((p.S & 3) | (p.H & 3) | (int)(reinterpret_cast<uintptr_t>(p.onehot) & 15)) == 0) for (int i = 0; i < p.S; i += 4) cp16(stage_at(r, p.H + i), src + i);
                else for (int i = 0; i < p.S; ++i) cp4(stage_at(r, p.H + i), src + i);
            } else if (cq == 2 && p.mode == 2) {
                const float* xj = p.x + (size_t)jet * p.N * 3;
                const int near = t->seg_near[sgq];
                for (int i = 0; i < 3; ++i) { cp4(stage_at(r, p.H + p.S + i), xj + slot * 3 + i); cp4(stage_at(r, p.H + p.S + 3 + i), xj + near * 3 + i); }
            }
        }
        if (cq == 3) {
            for (int sg = 0; sg < t->n_seg; ++sg) {
                const float* tb = p.tbias + (size_t)t->seg_jet[sg] * p.tbias_stride;
                for (int i = r; i < nblk * (kC / 4); i += 128) cp16(sTbias + sg * nblk * kC + 4 * i, tb + 4 * i);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if ((int)blockIdx.x < n_tiles) {   // the first tile of this CTA: all steps at once
        desc_issue(blockIdx.x);
        desc_commit(tn);
        __syncthreads();
        masks_issue(tn);
        rowmap_build(tn);
        __syncthreads();
        rows_prefetch(tn);
    }
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
        { TileState* tmp = ts; ts = tn; tn = tmp; }
        const int next_tile = tile + (int)gridDim.x;
        const bool has_next = next_tile < n_tiles;
        if (has_next) desc_issue(next_tile);
        seg = ts->qseg[qq];
        seg_first = seg >= 0 ? ts->seg_q0[seg] : qq;
        seg_nq = seg >= 0 ? ts->seg_nq[seg] : 1;
        w_row = ts->w[r];
        const int slot = ts->slot[r];
        // ---- proj_in: mode 0 [hidden, one_hot(mask)] (absorbing_flows.py:113-118); mode 1 [hidden, onehot]
        //      (transdimensional_model.py:295-303); mode 2 mask * [hidden, onehot, distance to the nearest particle,
        //      its one-hot flag pair] (transdimensional_model.py:341-367)
        if (cq == 0) {
            // the staged row already is [hidden | onehot | ...]: eight 16-byte reads at compile-time register positions (a row[]
            // indexed by H would live in local memory), then the mode's extra columns selected in
            float row[32];
            const float4* st4 = reinterpret_cast<const float4*>(sStage + r * 32);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 t4 = st4[c ^ (r & 7)];
                row[4 * c] = t4.x; row[4 * c + 1] = t4.y; row[4 * c + 2] = t4.z; row[4 * c + 3] = t4.w;
            }
            const int H = p.H, W0 = p.mode == 0 ? H : H + p.S;   // columns copied as they are
            float e0 = 0.0f, e1 = 0.0f, e2 = 0.0f;               // columns W0, W0 + 1, W0 + 2
            bool zero_all = slot < 0;
            if (slot >= 0) {
                const int m = (ts->mbits[seg][slot >> 5] >> (slot & 31)) & 1u;
                if (p.mode == 0) {
                    e0 = m ? 0.0f : 1.0f;
                    e1 = m ? 1.0f : 0.0f;
                } else if (p.mode == 2) {
                    const int near = ts->seg_near[seg];
                    const float d0 = *stage_at(r, W0 + 3) - *stage_at(r, W0), d1 = *stage_at(r, W0 + 4) - *stage_at(r, W0 + 1),
                                d2 = *stage_at(r, W0 + 5) - *stage_at(r, W0 + 2);
                    e0 = sqrtf((d0 * d0 + d1 * d1) + d2 * d2);
                    e1 = slot == near ? 1.0f : 0.0f;
                    e2 = slot == near ? 0.0f : 1.0f;
                    zero_all = !m;
                }
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {   // selects, never arithmetic: stale staging bytes beyond the row's width may be anything
                const float val = i < W0 ? row[i] : i == W0 ? e0 : i == W0 + 1 ? e1 : i == W0 + 2 ? e2 : 0.0f;
                row[i] = zero_all ? 0.0f : val;
            }
            uint8_t* q = sA0 + (r >> 3) * 512 + (r & 7) * 16;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(q + c * 128) = make_uint4(pack_bf16(row[8 * c], row[8 * c + 1]), pack_bf16(row[8 * c + 2], row[8 * c + 3]),
                                                                    pack_bf16(row[8 * c + 4], row[8 * c + 5]), pack_bf16(row[8 * c + 6], row[8 * c + 7]));
        } else {   // conv1 bias + the time term of every block, per jet of the tile
            for (int i = tid - 128; i < ts->n_seg * nblk * kC; i += kThreads - 128) {
                const int c = i % (nblk * kC);
                s_bias2[i] = sTab[(c >> 7) * HeadTable::kPerBlock + 2 * kC + (c & 127)] + sTbias[i];
            }
        }
        tc_fence_before();
        fence_proxy_async();
        __syncthreads();
        mma_issue([&](uint32_t ws) { gemm_w(ws, dX, smem_u32(sA0), 512, 2, false, true, bar_mma); });
        mma_done(1);
        const float* bias2 = s_bias2 + (seg < 0 ? 0 : seg) * nblk * kC;

        for (int blk = 0; blk < nblk; ++blk) {
            const float* T = sTab + blk * HeadTable::kPerBlock;
            // ---- ResnetBlock (gsdm.py:54-66)
            group_norm_to_A(dX, nullptr, T + 0 * kC, T + 1 * kC, true);
            mma_issue([&](uint32_t ws) { gemm_w(ws, dACC, aA, 2048, 8, false, false, bar_mma); });           // conv1
            if (blk == 0 && has_next) desc_commit(tn);       // next tile's preparation rides under the GEMM round trips
            mma_done(1);
            group_norm_to_A(dACC, bias2 + blk * kC, T + 3 * kC, T + 4 * kC, true);
            mma_issue([&](uint32_t ws) { gemm_w(ws, dX, aA, 2048, 8, true, true, bar_mma); });               // X += conv2(.) + b2
            if (blk == 0 && has_next) masks_issue(tn);
            mma_done(1);
            // ---- AttnBlock (gsdm.py:142-168)
            group_norm_to_A(dX, nullptr, T + 5 * kC, T + 6 * kC, false);
            const uint32_t q_half = wseq & 1;                                // q sits in ring slot wseq & 1
            mma_issue([&](uint32_t ws) { gemm_qk(ws, dACC, aA); });                                 // [q | k] (+ bq), one N = 256 GEMM into ACC | S0
            if (blk == 0 && has_next) rowmap_build(tn);
            mma_done(2);
            {   // both tiles in one epilogue phase
                float v[CW];
                tmem_ld32(dACC + q_half * 128 + lane_off + col0, v);
                store_row<CW>(sQ, r, col0, v);
                tmem_ld32(dACC + (q_half ^ 1) * 128 + lane_off + col0, v);
                store_row<CW>(sK, r, col0, v);
                tc_fence_before();
                fence_proxy_async();
                __syncthreads();
            }
            mma_issue([&](uint32_t ws) {                                     // S_h = Q_h K_h^T, K = 64
                tc_fence_after();
                const uint64_t qd = smem_desc(aQ, 128, 2048), kd = smem_desc(aK, 128, 2048);
#pragma unroll
                for (int h = 0; h < kHeads; ++h)
#pragma unroll
                    for (int j = 0; j < 4; ++j)   // head h = K-steps 4h .. 4h+3 of the Q and K tiles (1024 B = 64 in the address field)
                        umma(h ? dS1 : dS0, qd + (uint64_t)(h * 64 + j * 16), kd + (uint64_t)(h * 64 + j * 16), idesc128, j > 0);
                umma_commit(bar_mma);
                gemm_w(ws, dACC, aA, 2048, 8, false, false, bar_mma2);        // v: runs under the softmax, its own barrier
            });
            mma_done(0);
            // softmax over the keys of the query's OWN jet (block-diagonal): thread (r, cq) serves head cq / HQ and the two 32-key
            // chunks (= row quarters) 2 (cq % HQ), 2 (cq % HQ) + 1; a chunk of another jet contributes nothing, a key's column
            // of P carries the key's row weight (the representative dead row stands for n_dead identical keys).  The HQ threads
            // of a (row, head) exchange max and sum through shared memory.  P (unnormalised, bf16) -> K tile (head 0) / Q tile
            // (head 1), both dead once S is complete; the A tile still feeds the v GEMM.
            const int h = cq / HQ, key0 = (cq % HQ) * 2 * CW;
            {
                const uint32_t dS = (h ? dS1 : dS0) + lane_off + key0;
                float v[CW], mx = -3.0e38f;
                uint32_t mine = 0, weighted = 0;   // bit c: chunk c (registers: an array indexed by the rolled loop would live in local memory)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int kq = key0 / CW + c;                      // the chunk's row quarter
                    const bool mc = seg >= 0 && ts->qseg[kq] == seg;
                    mine |= (mc ? 1u : 0u) << c;
                    weighted |= (mc && ts->qwt[kq] ? 1u : 0u) << c;
                }
#pragma unroll 1
                for (int c = 0; c < 2; ++c) {
                    if (!((mine >> c) & 1u)) continue;
                    tmem_ld32(dS + c * CW, v);
                    if ((weighted >> c) & 1u) {   // keys of weight 0 (unused rows) leave the maximum: + (-3e38)
#pragma unroll
                        for (int j = 0; j < CW; j += 4) {
                            const float4 b4 = *reinterpret_cast<const float4*>(&ts->kb[key0 + c * CW + j]);
                            fadd2(v[j], v[j + 1], v[j], v[j + 1], b4.x, b4.y);
                            fadd2(v[j + 2], v[j + 3], v[j + 2], v[j + 3], b4.z, b4.w);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < CW; j += 2) mx = fmaxf(mx, fmaxf(v[j], v[j + 1]));
                }
                s_rowx[cq][r] = mx;
                named_bar(1 + NQ + h, 128 * HQ);   // the key slices of a head
#pragma unroll
                for (int i = 0; i < HQ; ++i) mx = fmaxf(mx, s_rowx[h * HQ + i][r]);
                const float sc = 0.125f * 1.4426950408889634f;  // dh^-1/2 * log2(e)
                const float off = -mx * sc;
                float s0 = 0.0f, s1 = 0.0f;
#pragma unroll 1
                for (int c = 0; c < 2; ++c) {
                    if ((mine >> c) & 1u) {
                        tmem_ld32(dS + c * CW, v);
                        if ((weighted >> c) & 1u) {   // P_j = w_j exp(.) = exp2(. + log2 w_j); w_j = 0 -> exp2(-inf) = 0
#pragma unroll
                            for (int j = 0; j < CW; j += 4) {
                                float4 l4 = *reinterpret_cast<const float4*>(&ts->lw[key0 + c * CW + j]);
                                fadd2(l4.x, l4.y, l4.x, l4.y, off, off);
                                fadd2(l4.z, l4.w, l4.z, l4.w, off, off);
                                ffma2(v[j], v[j + 1], v[j], v[j + 1], sc, sc, l4.x, l4.y);
                                ffma2(v[j + 2], v[j + 3], v[j + 2], v[j + 3], sc, sc, l4.z, l4.w);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < CW; j += 2) ffma2(v[j], v[j + 1], v[j], v[j + 1], sc, sc, off, off);
                        }
#pragma unroll
                        for (int j = 0; j < CW; j += 2) {
                            v[j] = ex2_fast(v[j]);
                            v[j + 1] = ex2_fast(v[j + 1]);
                            fadd2(s0, s1, s0, s1, v[j], v[j + 1]);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < CW; ++j) v[j] = 0.0f;
                    }
                    store_row<CW>(h ? sQ : sK, r, key0 + c * CW, v);
                }
                s_sum[cq][r] = s0 + s1;
                // the v GEMM finished long ago: its tile joins this phase's fence and barrier
                mbar_wait(bar_mma2, mma2_phase); mma2_phase ^= 1;
                tc_fence_after();
                if (tid == 0 && wseq + 2 < total_mats) issue_load(wseq + 2);
                ++wseq;
                tmem_ld32(dACC + lane_off + col0, v);
                if (seg < 0) {
#pragma unroll
                    for (int j = 0; j < CW; ++j) v[j] = 0.0f;     // V rows of an empty quarter meet zero columns of P, but 0 x NaN is NaN
                }
                store_row<CW>(sV, r, col0, v);
            }
            tc_fence_before();
            fence_proxy_async();
            __syncthreads();
            mma_issue([&](uint32_t) {                                        // O_h = P_h V_h, K = 128 keys, N = 64
                tc_fence_after();
                const uint64_t vd = smem_desc(aV, 2048, 128);
#pragma unroll
                for (int hh = 0; hh < kHeads; ++hh) {
                    const uint64_t pd = smem_desc(hh ? aQ : aK, 128, 2048);
#pragma unroll
                    for (int j = 0; j < 8; ++j)   // V MN-major: head hh starts 1024 B in, a K-step of 16 keys is 4096 B
                        umma(dACC + hh * 64, pd + (uint64_t)(j * 16), vd + (uint64_t)(hh * 64 + j * 256), idesc64mn, j > 0);
                }
                umma_commit(bar_mma);
            });
            mma_done(0);
            if (blk == nblk - 1 && has_next) rows_prefetch(tn);   // V is dead now
            {
                float v[CW];  // columns [col0, +CW) of O belong to head cq / HQ: normalised by that head's row sum
                float tot = 0.0f;
#pragma unroll
                for (int i = 0; i < HQ; ++i) tot += s_sum[h * HQ + i][r];
                const float rinv = tot > 0.0f ? 1.0f / tot : 0.0f;    // empty quarter: no keys
                tmem_ld32(dACC + lane_off + col0, v);
#pragma unroll
                for (int j = 0; j < CW; j += 2) fmul2(v[j], v[j + 1], v[j], v[j + 1], rinv, rinv);
                store_row<CW>(sA, r, col0, v);
            }
            tc_fence_before();
            fence_proxy_async();
            __syncthreads();
            mma_issue([&](uint32_t ws) { gemm_w(ws, dX, aA, 2048, 8, true, true, bar_mma); });               // X += proj_out(.) + (b_o + W_o b_v)
            mma_done(1);
        }
        // ---- per-slot output: one 128-vector against the residual stream (absorbing: post_rate_proj(pre_rate_proj(X))
        //      folded, absorbing_flows.py:127-131; trans: near_atom_proj / vec_weighting_proj) and, for the per-jet heads,
        //      the mean of X over the N slots (transdimensional_model.py:309-311,403-405; the folded Linear follows in jet_head_kernel)
        {
            const float* w = sTab + HeadTable::rate_w(nblk);
            float v[CW], a0 = 0.0f, a1 = 0.0f;
            tmem_ld32(dX + lane_off + col0, v);
#pragma unroll
            for (int j = 0; j < CW; j += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(w + col0 + j);
                ffma2(a0, a1, v[j], v[j + 1], w4.x, w4.y, a0, a1);
                ffma2(a0, a1, v[j + 2], v[j + 3], w4.z, w4.w, a0, a1);
            }
            s_dot[cq][r] = a0 + a1;
            if (p.n_jet > 0) {   // weighted column sums over the rows: halving reduction inside the warp, then the jet's quarters
#pragma unroll
                for (int j = 0; j < CW; ++j) v[j] = w_row > 0.0f ? v[j] * w_row : 0.0f;
                warp_halving_sum<CW>(v, lane);
                if ((lane & (32 / CW - 1)) == 0) s_part[warp][warp_halving_index<CW>(lane)] = v[0];
            }
            __syncthreads();
            // every slot of every jet of the tile gets its value: a live slot from its own row, a padded slot from the jet's
            // representative row
            for (int it = tid; it < ts->n_seg * p.N; it += kThreads) {
                const int sg = it / p.N, n = it - sg * p.N;
                const int m = ts->seg_m[sg], base = 32 * ts->seg_q0[sg];
                int row;
                if (!ts->seg_packed[sg]) row = base + n;
                else if ((ts->mbits[sg][n >> 5] >> (n & 31)) & 1u) {
                    int below = __popc(ts->mbits[sg][n >> 5] & ((1u << (n & 31)) - 1u));
                    for (int wd = 0; wd < (n >> 5); ++wd) below += __popc(ts->mbits[sg][wd]);
                    row = base + below;
                } else row = base + m;
                float tot = sTab[HeadTable::rate_c(nblk)];
#pragma unroll
                for (int i = 0; i < NQ; ++i) tot += s_dot[i][row];
                p.logit_out[(size_t)ts->seg_jet[sg] * p.N + n] = tot;
            }
            if (p.n_jet > 0 && tid < 128) {   // the folded per-jet Linear runs afterwards, batched over jets (jet_head_kernel)
                const int w0 = (tid / CW) * 4, ci = tid % CW;
                for (int sg = 0; sg < ts->n_seg; ++sg) {
                    float sum = 0.0f;
                    for (int i = 0; i < ts->seg_nq[sg]; ++i) sum += s_part[w0 + ts->seg_q0[sg] + i][ci];
                    p.jet_out[(size_t)ts->seg_jet[sg] * kC + tid] = sum * (1.0f / (float)p.N);
                }
            }
        }
        tc_fence_before();
        __syncthreads();  // X, the operand tiles and the tile's tables are rewritten by the next tile
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace

// ---- host side: one transformer stack = operand image + side table (+ optional per-jet head) --------------------------
void tf_stack_free(TfStack* st) {
    if (st->image) cudaFree(st->image);
    if (st->table) cudaFree(st->table);
    if (st->jet_wT) cudaFree(st->jet_wT);
    if (st->jet_b) cudaFree(st->jet_b);
    *st = TfStack{};
}

// proj_in [C][Cin]+[C]; blocks: n_blocks x (norm1 g b, conv1, norm2 g b, conv2, attn norm g b, q, k, v, proj_out), every conv
// [C][C]+[C]; dot_w [C] / dot_c: the per-particle output; jet_w [n_jet][C] / jet_b [n_jet]: the per-jet head (nullable).
// Allocates on the CURRENT device.
int tf_stack_build(TfStack* st, const float* proj_in, int Cin, const float* blocks, int n_blocks, const float* dot_w, float dot_c,
                   const float* jet_w, const float* jet_b, int n_jet) {
    constexpr int C = kC;
    if (n_blocks < 1 || n_blocks > kMaxBlocks || Cin < 1 || Cin > 32 || n_jet < 0 || n_jet > 128)
        return fail(MMB_EUNSUPPORTED, "transformer stack is built for 1..4 blocks, <= 32 input features, <= 128 per-jet outputs");
    const size_t lin = (size_t)C * C + C;
    const int n_seq = 1 + 6 * n_blocks;
    std::vector<__nv_bfloat16> img((size_t)n_seq * kSlot / 2, __float2bfloat16(0.0f));
    std::vector<float> tab((size_t)HeadTable::floats(n_blocks), 0.0f);
    auto put_matrix = [&](int slot, const float* Wm, int in_dim) {
        for (int o = 0; o < C; ++o)
            for (int k = 0; k < in_dim; ++k) slot_put_weight(img, slot, o, k, Wm[(size_t)o * in_dim + k]);
    };
    auto put_bias = [&](int slot, const float* b) {
        for (int o = 0; o < C; ++o) slot_put_bias(img, slot, o, b[o]);
    };
    put_matrix(0, proj_in, Cin);
    put_bias(0, proj_in + (size_t)C * Cin);
    const float* p = blocks;
    for (int blk = 0; blk < n_blocks; ++blk) {
        float* T = tab.data() + (size_t)blk * HeadTable::kPerBlock;
        const float *n1g = p, *n1b = p + C, *c1 = p + 2 * C, *n2g = c1 + lin, *n2b = n2g + C, *c2 = n2b + C, *ng = c2 + lin,
                    *nb = ng + C, *wq = nb + C, *wk = wq + lin, *wv = wk + lin, *wo = wv + lin;
        p = wo + lin;
        const int s0 = 1 + 6 * blk;
        put_matrix(s0 + 0, c1, C);
        put_matrix(s0 + 1, c2, C); put_bias(s0 + 1, c2 + (size_t)C * C);
        put_matrix(s0 + 2, wq, C); put_bias(s0 + 2, wq + (size_t)C * C);
        put_matrix(s0 + 3, wk, C);          // k bias: a per-query constant in the logits, softmax-invariant
        put_matrix(s0 + 4, wv, C);          // v bias: softmax rows sum to one -> O gains b_v, i.e. proj_out gains W_o b_v
        put_matrix(s0 + 5, wo, C);
        {
            std::vector<float> bo(C);
            const float* bv = wv + (size_t)C * C;
            for (int o = 0; o < C; ++o) {
                double acc = wo[(size_t)C * C + o];
                for (int c = 0; c < C; ++c) acc += (double)wo[(size_t)o * C + c] * bv[c];
                bo[o] = (float)acc;
            }
            put_bias(s0 + 5, bo.data());
        }
        for (int c = 0; c < C; ++c) {
            T[0 * kC + c] = n1g[c]; T[1 * kC + c] = n1b[c]; T[2 * kC + c] = c1[(size_t)C * C + c];
            T[3 * kC + c] = n2g[c]; T[4 * kC + c] = n2b[c]; T[5 * kC + c] = ng[c]; T[6 * kC + c] = nb[c];
        }
    }
    for (int c = 0; c < C; ++c) tab[HeadTable::rate_w(n_blocks) + c] = dot_w[c];
    tab[HeadTable::rate_c(n_blocks)] = dot_c;
    *st = TfStack{};
    st->Cin = Cin; st->n_blocks = n_blocks; st->n_jet = n_jet;
    int rc = cuda_ok(cudaMalloc(&st->image, img.size() * 2), "cudaMalloc stack image");
    if (!rc) rc = cuda_ok(cudaMalloc(&st->table, tab.size() * 4), "cudaMalloc stack table");
    if (!rc) rc = cuda_ok(cudaMemcpy(st->image, img.data(), img.size() * 2, cudaMemcpyHostToDevice), "stack image upload");
    if (!rc) rc = cuda_ok(cudaMemcpy(st->table, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice), "stack table upload");
    if (!rc && n_jet > 0) {
        std::vector<float> wT((size_t)C * n_jet);
        for (int o = 0; o < n_jet; ++o)
            for (int c = 0; c < C; ++c) wT[(size_t)c * n_jet + o] = jet_w[(size_t)o * C + c];
        rc = cuda_ok(cudaMalloc(&st->jet_wT, wT.size() * 4), "cudaMalloc jet head");
        if (!rc) rc = cuda_ok(cudaMalloc(&st->jet_b, (size_t)n_jet * 4), "cudaMalloc jet head bias");
        if (!rc) rc = cuda_ok(cudaMemcpy(st->jet_wT, wT.data(), wT.size() * 4, cudaMemcpyHostToDevice), "jet head upload");
        if (!rc) rc = cuda_ok(cudaMemcpy(st->jet_b, jet_b, (size_t)n_jet * 4, cudaMemcpyHostToDevice), "jet head bias upload");
    }
    if (rc) tf_stack_free(st);
    return rc;
}

// Per-jet head: out[b][o] = bias[o] + sum_c W^T[c][o] * mean[b][c], batched so that every weight row is read once per 16 jets.
__global__ void __launch_bounds__(128) jet_head_kernel(const float* __restrict__ means, const float* __restrict__ wT, const float* __restrict__ bias,
                                                       int n_out, int B, float* __restrict__ out) {
    constexpr int JB = 16;
    __shared__ __align__(16) float s_m[kC][JB];   // [channel][jet]: one LDS.128 serves four jets
    const int o = threadIdx.x, j0 = blockIdx.x * JB;
    for (int i = threadIdx.x; i < JB * kC; i += 128) {
        const int j = i / kC, c = i % kC;
        s_m[c][j] = j0 + j < B ? __ldg(means + (size_t)(j0 + j) * kC + c) : 0.0f;
    }
    __syncthreads();
    if (o >= n_out) return;
    float acc[JB];
    const float b = __ldg(bias + o);
#pragma unroll
    for (int j = 0; j < JB; ++j) acc[j] = b;
#pragma unroll 8
    for (int c = 0; c < kC; ++c) {
        const float w = __ldg(wT + (size_t)c * n_out + o);
#pragma unroll
        for (int j = 0; j < JB; j += 4) {
            const float4 m4 = *reinterpret_cast<const float4*>(&s_m[c][j]);
            acc[j] = fmaf(w, m4.x, acc[j]); acc[j + 1] = fmaf(w, m4.y, acc[j + 1]);
            acc[j + 2] = fmaf(w, m4.z, acc[j + 2]); acc[j + 3] = fmaf(w, m4.w, acc[j + 3]);
        }
    }
#pragma unroll
    for (int j = 0; j < JB; ++j)
        if (j0 + j < B) out[(size_t)(j0 + j) * n_out + o] = acc[j];
}

int launch_jet_head(const TfStack* st, const float* means, int B, float* out, cudaStream_t stream) {
    if (B == 0 || st->n_jet == 0) return MMB_OK;
    jet_head_kernel<<<(B + 15) / 16, 128, 0, stream>>>(means, st->jet_wT, st->jet_b, st->n_jet, B, out);
    return cuda_ok(cudaGetLastError(), "jet head launch");
}

int launch_tf_stack(const TfStack* st, int sm_count, const TfStackIO& io, int B, int N, cudaStream_t stream) {
    if (N < 1 || N > 128) return fail(MMB_EUNSUPPORTED, "transformer stack handles 1..128 particle slots per jet (got %d)", N);
    if (B == 0) return MMB_OK;
    HeadParams p{};
    p.image = static_cast<const uint8_t*>(st->image); p.table = st->table; p.n_blocks = st->n_blocks; p.H = io.H;
    p.mode = io.mode; p.S = io.S; p.hidden = io.hidden; p.mask = io.mask; p.onehot = io.onehot; p.x = io.x; p.nearest = io.nearest;
    p.tbias = io.tbias; p.tbias_stride = io.tbias_stride; p.B = B; p.N = N; p.logit_out = io.dot_out;
    p.n_jet = io.jet_out ? st->n_jet : 0; p.jet_out = io.jet_out;
    if (io.pack_scratch) {   // bin the jets by the quarters of a tile they need (dead slots once, several jets per tile)
        if (io.pack_scratch_ints < PackScratch::ints(B)) return fail(MMB_ENOMEM, "transformer stack: packing scratch too small");
        if (int rc = cuda_ok(cudaMemsetAsync(io.pack_scratch, 0, 8 * sizeof(int32_t), stream), "pack counters")) return rc;
        tf_pack_kernel<<<(B + 7) / 8, 256, 0, stream>>>(io.mask, io.hidden, io.H, io.onehot, io.S, io.mode, B, N, io.pack_scratch);
        tf_tiles_kernel<<<(B + 255) / 256, 256, 0, stream>>>(io.pack_scratch, B);
        if (int rc = cuda_ok(cudaGetLastError(), "tf_pack launch")) return rc;
        p.pack = io.pack_scratch;
    }
    const size_t bytes = kOffTab + (size_t)(HeadTable::floats(st->n_blocks) + kMaxSeg * st->n_blocks * kC) * 4;
    auto kern = absorb_head_tc_kernel;
    cudaFuncAttributes attr;
    if (int rc = cuda_ok(cudaFuncGetAttributes(&attr, kern), "head attributes")) return rc;
    if (bytes + attr.sharedSizeBytes > 232448)
        return fail(MMB_EUNSUPPORTED, "transformer stack with %d blocks needs %zu B of shared memory per CTA (limit 232448)", st->n_blocks,
                    bytes + attr.sharedSizeBytes);
    if (int rc = cuda_ok(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), "head smem attribute"))
        return rc;
    const int grid = B < sm_count ? B : sm_count;
    kern<<<grid, kThreads, bytes, stream>>>(p);
    return cuda_ok(cudaGetLastError(), "transformer stack launch");
}

struct AbsorbHead {
    int H, C, n_heads, n_blocks, device, sm_count;
    TfStack stack;
};

int absorb_head_create(int H, int C, int n_heads, int n_blocks, const float* W, size_t n_floats, int device, AbsorbHead** out) {
    if (C != kC || n_heads != kHeads || n_blocks < 1 || n_blocks > kMaxBlocks || H < 1 || H > 30)
        return fail(MMB_EUNSUPPORTED, "absorbing head is built for transformer_dim=128, n_heads=2, 1..4 blocks, hidden<=30");
    const size_t lin = (size_t)C * C + C;
    const size_t expect = (size_t)C * (H + 2) + C + (size_t)n_blocks * (6 * C + 6 * lin) + lin + C + 1;
    if (n_floats != expect) return fail(MMB_EINVAL, "absorbing head blob has %zu floats, layout wants %zu", n_floats, expect);
    const float* blocks = W + (size_t)C * (H + 2) + C;
    const float* p = blocks + (size_t)n_blocks * (6 * C + 6 * lin);
    // fold Linear(C->C) then Linear(C->1): w = post^T pre, c = post . pre_b + post_b
    std::vector<float> dot_w(C);
    const float *pre = p, *pre_b = p + (size_t)C * C, *post = p + lin, *post_b = post + C;
    for (int c = 0; c < C; ++c) {
        double acc = 0;
        for (int o = 0; o < C; ++o) acc += (double)post[o] * pre[(size_t)o * C + c];
        dot_w[c] = (float)acc;
    }
    double dc = post_b[0];
    for (int o = 0; o < C; ++o) dc += (double)post[o] * pre_b[o];
    int prev = 0;
    if (int rc = cuda_ok(cudaGetDevice(&prev), "cudaGetDevice")) return rc;
    if (int rc = cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return rc;
    AbsorbHead* h = new AbsorbHead{H, C, n_heads, n_blocks, device, 148, TfStack{}};
    int rc = cuda_ok(cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device), "sm count");
    if (!rc) rc = tf_stack_build(&h->stack, W, H + 2, blocks, n_blocks, dot_w.data(), (float)dc, nullptr, nullptr, 0);
    cudaSetDevice(prev);
    if (rc) { delete h; return rc; }
    *out = h;
    return MMB_OK;
}

void absorb_head_destroy(AbsorbHead* h) {
    if (!h) return;
    tf_stack_free(&h->stack);
    delete h;
}

int absorb_head_hidden(const AbsorbHead* h) { return h->H; }
int absorb_head_blocks(const AbsorbHead* h) { return h->n_blocks; }

size_t tf_pack_scratch_ints(int B) { return PackScratch::ints(B > 0 ? B : 0); }

int launch_absorb_head(const AbsorbHead* h, const float* hidden, const uint8_t* mask, const float* tbias, int tbias_stride,
                       int B, int N, float* logit_out, cudaStream_t stream, int32_t* pack_scratch, size_t pack_scratch_ints) {
    TfStackIO io{};
    io.mode = 0; io.H = h->H; io.hidden = hidden; io.mask = mask; io.tbias = tbias; io.tbias_stride = tbias_stride; io.dot_out = logit_out;
    io.pack_scratch = pack_scratch; io.pack_scratch_ints = pack_scratch_ints;
    return launch_tf_stack(&h->stack, h->sm_count, io, B, N, stream);
}

}  // namespace mmb
