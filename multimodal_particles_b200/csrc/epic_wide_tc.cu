// epic_wide_tc.cu — EPiC with 128 hidden units per particle on tcgen05 tensor cores (sm_100a).
//
// The class default of the reference's EPiCNetwork is dim_hidden_local = 128, num_blocks = 6 (mp/models/architectures/epic.py:
// 99-101); at that width a network evaluation is real GEMM work: per EPiC layer two [N particles x 128] x [128 x 128] products
// (fc_local1, fc_local2: epic.py:233-238), 0.41 MFLOP per particle and evaluation at L = 6.  This file is the trunk for such
// models (`mmb_epic_forward` / the step loop of `mmb_generate` with MMB_PREC_BF16); the H = 16 engines live in epic_tc.cu /
// epic_mma.cu.
//
// One CTA (512 threads) carries TWO tiles at a time (A and B, 128 rows each = TMEM lanes), persistent over pairs of tiles.  Rows are
// LIVE particles only: every per-particle layer acts on rows independently and the pooling is masked, so padded slots need no row
// at all (their outputs are constants, written by the pre-pass).  A jet takes ceil(live / 32) of a tile's four 32-row quarters and
// a tile holds one or two jets (pre-pass: wide_pack_kernel bins the jets, wide_tiles_kernel composes [4] | [3,1] | [2,2] | [2,1] |
// [1,1]), so a CTA works on up to four jets:
//   * per tile the residual stream X [128 x 128] fp32 and one accumulator ACC [128 x 128] live in TMEM (2 x 256 = all 512 columns);
//     thread (r, cq) serves row r, columns [32 cq, 32 cq + 32) of whichever tile is in its epilogue;
//   * every Linear over the particles is 8 tcgen05.mma M128 x N128 x K16 with bf16 operands; the weights stream L2 -> shared
//     memory by 1-D TMA into a two-slot ring, one matrix ahead, and each matrix serves both tiles;
//   * the two tiles are staggered: while the CUDA cores run the epilogue of one (bias, leaky-ReLU, mask, skip, pooling sums,
//     bf16 operand for the next GEMM, fp32 residual back to TMEM with tcgen05.st), the tensor core runs the GEMM of the other;
//   * fc_local2 accumulates straight onto X (the residual add is the accumulate flag), its bias rides on one more K-step
//     against a ones tile; fc_local1's bias is per jet (its global and context columns) and is added in the epilogue;
//   * local_0 with the embeddings folded in is ONE K-step: the operand row is [x_hi, x_lo, onehot(k)] (two bf16 per feature);
//   * the per-jet global path (masked mean / sum pooling -> global MLPs, epic.py:136-143, 187-190, 226-232) is warp-level
//     tensor-core work too: the jets of the CTA are the rows of mma.sync m16n8k16 tiles (inputs split into bf16 hi + lo, so they
//     enter with ~16 bits — except the 256 pooled features, plain bf16 like every particle activation), each of the 16 warps owns
//     eight output columns and reads its weight fragments, pre-arranged on the
//     host, straight from L2 — once per CTA and layer, while the fc_local1 GEMMs are in flight;
//   * the trunk skip (epic.py:148-155) is kept per tile as fp16 in shared memory.
// Numerics: bf16 operands (weights of both paths), fp32 accumulation, fp32 residual stream, pooling sums and biases.  Checked against the fp32 kernel with the tolerance written in tests/test_gpu_wide.py.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <vector>

#include "mmb_device.cuh"
#include "mmb_internal.h"
#include "tcgen05.cuh"

namespace mmb {
namespace {

constexpr int kH = 128;
constexpr int kThreads = 512;
constexpr int kCW = 32;             // accumulator columns per thread
constexpr int kMaxL = 8;

// 32 consecutive fp32 columns of this thread's TMEM lane: store
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
          "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
          "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
          "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
          "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// skip tile: fp16 [128 rows][128 cols], 256 B per row, 16-byte chunks XOR-swizzled by the row so that a quarter-warp (8 rows,
// same chunk number) touches 8 different bank groups
__device__ __forceinline__ uint4* skip_chunk(uint8_t* tile, int row, int chunk) {
    return reinterpret_cast<uint4*>(tile + row * 256 + ((chunk ^ (row & 7)) << 4));
}
__device__ __forceinline__ float lrelu(float a) { return a > 0.0f ? a : 0.01f * a; }
__device__ __forceinline__ float selu(float a) {
    const float alpha = 1.6732632423543772848170429916717f, scale = 1.0507009873554804934193349852946f;
    return scale * (a > 0.0f ? a : alpha * (__expf(a) - 1.0f));
}

__host__ __device__ inline int round16(int v) { return (v + 15) & ~15; }

constexpr int kMaxJ = 4;                 // jets per CTA: two tiles x two segments
constexpr int kMaxTXq = 64, kMaxGq = 32; // padded widths of the context vector [time | context] and of the global vector
constexpr int kIn1Stride = (256 + kMaxTXq + kMaxGq) / 2 + 4;   // words per jet of the fc_global1 input (bf16 pairs); = 20 mod 32
constexpr int kGvStride = 64 + 4;                              // a 128-vector; = 4 mod 32
constexpr int kCxStride = (kMaxTXq + kMaxGq) / 2 + 4;          // [ctx | xm]; = 20 mod 32
static_assert(kIn1Stride % 32 == 20 && kGvStride % 32 == 4 && kCxStride % 32 == 20, "row strides chosen so that (jet, t) lanes hit distinct banks");

// fp32 side table (floats) and the weight fragments of the global path (uint2 per lane, see put_frag)
struct WideLayout {
    int L, G, T, X, S, Sh, Dc, skip;
    int TXq, Gq;                // padded to multiples of 16 (zero weights in the padding)
    // fp32 table
    int c0, b_g0, b_g1, b_g2;   // [128] local_0 bias (+ folded embedding bias), biases of global_0 / global_1 / global_2 [Gq]
    int layer0, layer_stride;   // per layer: b_lg1 [128] | b_lg2 [Gq] | b_l1 [128]
    int o_blg1, o_blg2, o_bl1;
    int head0, b_head0, head2, b_head2, dead_logits;   // [16][16], [16], [16][16], [16], [8]: logits of a padded slot = head(0)
    int tab_floats;
    // fragment image (uint2 units): a matrix occupies (N / 8) * (KS rounded up to even) * 32 entries
    int f_w0t, f_g0, f_g1, f_g2;
    int f_layer0, f_layer_stride, fo_wg1, fo_wg2, fo_wl1g;
    int frag_elems;
    int n_seq;                  // streamed matrices per evaluation: local_0, L x (fc_local1, fc_local2), output
    __host__ __device__ int KS_t() const { return TXq / 16; }
    __host__ __device__ int KS_0() const { return (256 + TXq) / 16; }
    __host__ __device__ int KS_1() const { return (256 + TXq + Gq) / 16; }
    __host__ __device__ int KS_2() const { return (TXq + Gq) / 16; }
};

WideLayout make_layout(const MmbEpicDims& d) {
    WideLayout w{};
    w.L = d.num_blocks; w.G = d.dim_hidden_glob; w.T = d.dim_time_emb; w.X = d.dim_context; w.S = d.vocab_size; w.Sh = d.disc_head_hidden;
    w.Dc = d.dim_continuous; w.skip = d.skip_connection;
    w.TXq = round16(w.T + w.X); w.Gq = round16(w.G);
    int o = 0;
    auto take = [&](int n) { const int at = o; o += (n + 3) & ~3; return at; };
    w.c0 = take(128); w.b_g0 = take(128); w.b_g1 = take(128); w.b_g2 = take(w.Gq);
    w.layer0 = o;
    {
        int p = 0;
        auto tk = [&](int n) { const int at = p; p += (n + 3) & ~3; return at; };
        w.o_blg1 = tk(128); w.o_blg2 = tk(w.Gq); w.o_bl1 = tk(128);
        w.layer_stride = p;
    }
    o += w.layer_stride * w.L;
    w.head0 = take(256); w.b_head0 = take(16); w.head2 = take(256); w.b_head2 = take(16); w.dead_logits = take(8);
    w.tab_floats = o;
    int f = 0;
    auto tf = [&](int n_out, int ks) { const int at = f; f += (n_out / 8) * ((ks + 1) & ~1) * 32; return at; };   // k-steps stored in pairs
    w.f_w0t = tf(128, w.KS_t()); w.f_g0 = tf(128, w.KS_0()); w.f_g1 = tf(128, 8); w.f_g2 = tf(w.Gq, 8);
    w.f_layer0 = f;
    {
        int p = 0;
        auto tk = [&](int n_out, int ks) { const int at = p; p += (n_out / 8) * ((ks + 1) & ~1) * 32; return at; };
        w.fo_wg1 = tk(128, w.KS_1()); w.fo_wg2 = tk(w.Gq, 8); w.fo_wl1g = tk(128, w.KS_2());
        w.f_layer_stride = p;
    }
    f += w.f_layer_stride * w.L;
    w.frag_elems = f;
    w.n_seq = 2 + 2 * w.L;
    return w;
}

// ---- packing pre-pass ------------------------------------------------------------------------------------------------------------
// scratch (int32): counts[8] ([q] = jets needing q quarters, q = 1..4; [5] = tiles) | lists[4][B] | tile records [B][kRec]
constexpr int kRec = 12;   // n_seg, then per segment: jet, q0, nq, m  (+ padding)
__host__ __device__ inline size_t pack_ints(int B) { return 8 + (size_t)B * 4 + (size_t)B * kRec; }

// warp per jet: live count -> list of its class; the heads of padded slots are constants and are written here (v = 0,
// logits = head(0): the reference applies the head to the masked logits, mbm.py:105-111; hidden = 0); a jet without particles is
// NaN throughout (its mean pool is 0 / 0, epic.py:141, and NaN * mask stays NaN) and is finished here
__global__ void __launch_bounds__(256) wide_pack_kernel(const uint8_t* __restrict__ mask, int B, int N, int S, const float* __restrict__ dead_logits,
                                                        float* __restrict__ v_out, float* __restrict__ logits_out, float* __restrict__ hidden_out,
                                                        int32_t* __restrict__ pack) {
    const int jet = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (jet >= B) return;
    int m = 0;
    for (int n0 = 0; n0 < N; n0 += 32) m += __popc(__ballot_sync(0xffffffffu, n0 + lane < N && mask[(size_t)jet * N + n0 + lane] != 0));
    const float nan = __int_as_float(0x7fc00000);
    for (int n = lane; n < N; n += 32) {
        if (mask[(size_t)jet * N + n]) continue;
        const size_t pi = (size_t)jet * N + n;
        for (int c = 0; c < 3; ++c) v_out[pi * 3 + c] = m ? 0.0f : nan;
        for (int s = 0; s < S; ++s) logits_out[pi * S + s] = m ? dead_logits[s] : nan;
        if (hidden_out)
            for (int c = 0; c < kH; c += 4) *reinterpret_cast<float4*>(hidden_out + pi * kH + c) = m ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(nan, nan, nan, nan);
    }
    if (lane == 0 && m > 0) {
        const int q = (m + 31) / 32;
        const int pos = atomicAdd(pack + q, 1);
        pack[8 + (size_t)B * (q - 1) + pos] = jet | (m << 20);
    }
}

// tiles: [4] x n4 | [3 (+1)] x n3 | [2,2] x n2/2 | [2 (+1)] if n2 is odd | [1,1] ...; one thread per tile
__global__ void __launch_bounds__(256) wide_tiles_kernel(int32_t* __restrict__ pack, int B) {
    const int n1 = pack[1], n2 = pack[2], n3 = pack[3], n4 = pack[4];
    const int32_t *l1 = pack + 8, *l2 = l1 + B, *l3 = l2 + B, *l4 = l3 + B;
    const int a = min(n3, n1), b = (n2 & 1) ? min(1, n1 - a) : 0;
    const int n_tiles = n4 + n3 + n2 / 2 + (n2 & 1) + (n1 - a - b + 1) / 2;
    if (blockIdx.x == 0 && threadIdx.x == 0) pack[5] = n_tiles;
    int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= n_tiles) return;
    int n_seg = 0, e[2] = {0, 0}, nq[2] = {0, 0};
    auto add = [&](int entry, int q) { e[n_seg] = entry; nq[n_seg] = q; ++n_seg; };
    if (t < n4) add(l4[t], 4);
    else if ((t -= n4) < n3) { add(l3[t], 3); if (t < a) add(l1[t], 1); }
    else if ((t -= n3) < n2 / 2) { add(l2[2 * t], 2); add(l2[2 * t + 1], 2); }
    else {
        t -= n2 / 2;
        if ((n2 & 1) && t == 0) { add(l2[n2 - 1], 2); if (b) add(l1[a], 1); }
        else {
            t -= (n2 & 1);
            add(l1[a + b + 2 * t], 1);
            if (a + b + 2 * t + 1 < n1) add(l1[a + b + 2 * t + 1], 1);
        }
    }
    int32_t* rec = pack + 8 + (size_t)B * 4 + (size_t)(blockIdx.x * 256 + threadIdx.x) * kRec;
    rec[0] = n_seg;
    for (int s = 0; s < 2; ++s) {
        rec[1 + 4 * s] = e[s] & 0xfffff; rec[2 + 4 * s] = s ? nq[0] : 0; rec[3 + 4 * s] = nq[s]; rec[4 + 4 * s] = e[s] >> 20;
    }
}

struct WideParams {
    const uint8_t* image;            // n_seq slots of kSlot bytes
    const float* tab;                // WideLayout fp32 table
    const uint2* frag;               // WideLayout weight fragments of the global path
    WideLayout lay;
    const int32_t* pack;             // pre-pass result
    const float* x;                  // [B,N,3]
    const uint8_t* k;                // [B,N]
    const uint8_t* mask;             // [B,N]
    const float* temb;               // [B or 1][T + X]
    int temb_stride;
    int B, N;
    float* v_out;                    // [B,N,3]
    float* logits_out;               // [B,N,S]
    float* hidden_out;               // [B,N,128] or null
};

// dynamic shared memory
constexpr int kOffRing = 0;
constexpr int kOffA = 2 * kSlot;                    // two operand tiles
constexpr int kOffSkip = kOffA + 2 * 32768;         // two fp16 skip tiles
constexpr int kOffOnes = kOffSkip + 2 * 32768;
constexpr int kOffVec = kOffOnes + 4096;            // per-jet vectors (4-byte words), see Vec
struct Vec {
    static constexpr int in1_hi = 0, in1_lo = in1_hi + kMaxJ * kIn1Stride;     // [mean 128 | sum 128 | ctx TXq | xg Gq] as bf16 pairs
    static constexpr int gva_hi = in1_lo + kMaxJ * kIn1Stride, gva_lo = gva_hi + kMaxJ * kGvStride;   // 128-vectors between the stages
    static constexpr int gvb_hi = gva_lo + kMaxJ * kGvStride, gvb_lo = gvb_hi + kMaxJ * kGvStride;
    static constexpr int cx_hi = gvb_lo + kMaxJ * kGvStride, cx_lo = cx_hi + kMaxJ * kCxStride;       // [ctx | xm]
    static constexpr int bl1 = cx_lo + kMaxJ * kCxStride;       // fp32 [kMaxJ][128]: per-jet bias of fc_local1 (of local_0 at tile start)
    static constexpr int xg = bl1 + kMaxJ * 128;                // fp32 [kMaxJ][32]
    static constexpr int skg = xg + kMaxJ * kMaxGq;             // fp32 [kMaxJ][32]
    static constexpr int part = skg + kMaxJ * kMaxGq;           // fp32 [2 tiles][16 warps][32]
    static constexpr int head = part + 2 * 16 * 32;             // head0 [16][16] | b0 [16] | head2 [16][16] | b2 [16]
    static constexpr int slot = head + 256 + 16 + 256 + 16;     // int [2 tiles][128]: row -> particle slot of its jet, -1 unused
    static constexpr int words = slot + 2 * 128;
};
constexpr int kSmemBytes = kOffVec + Vec::words * 4;
static_assert(kSmemBytes + 512 <= 227 * 1024, "shared memory budget");

template <int N>
struct FragRegs { uint2 b[N]; };   // weight fragments of one stage of the per-jet path, in registers

__device__ __forceinline__ void mma_bf16(float (&d)[4], uint32_t a0, uint32_t a2, const uint2 b) {   // rows 8..15 of A are zero
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(0u), "r"(a2), "r"(0u), "r"(b.x), "r"(b.y));
}
// fp32 pair -> bf16 pair words (hi, lo): value ~ hi + lo
__device__ __forceinline__ void split_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
    const float h0 = __bfloat162float(__float2bfloat16(v0)), h1 = __bfloat162float(__float2bfloat16(v1));
    hi = pack_bf16(h0, h1);
    lo = pack_bf16(v0 - h0, v1 - h1);
}

__global__ void __launch_bounds__(kThreads, 1) epic_wide_kernel(const WideParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t s_tmem_slot;
    __shared__ __align__(8) uint64_t s_bars[4];      // full[0], full[1], mma[A], mma[B]
    __shared__ int s_rec[2][kRec];                   // the two tiles of the pair
    __shared__ int s_qseg[2][4];                     // tile, quarter -> segment (-1: empty)
    const WideLayout& ly = p.lay;
    const int tid = threadIdx.x, r = tid & 127, cq = tid >> 7, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int qq = warp & 3, g = lane >> 2, t4 = lane & 3;
    const int L = ly.L, G = ly.G, Gq = ly.Gq, TXq = ly.TXq, TX = ly.T + ly.X, S = ly.S, Sh = ly.Sh;
    const bool skip_on = ly.skip != 0;
    uint8_t* sOnes = smem + kOffOnes;
    float* sv = reinterpret_cast<float*>(smem + kOffVec);
    uint32_t* sw = reinterpret_cast<uint32_t*>(smem + kOffVec);
    int* s_slot = reinterpret_cast<int*>(smem + kOffVec) + Vec::slot;
    auto sA = [&](int t) { return smem + kOffA + t * 32768; };
    auto sSkip = [&](int t) { return smem + kOffSkip + t * 32768; };

    for (int i = tid; i < 256; i += kThreads) reinterpret_cast<uint4*>(sOnes)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    for (int i = tid; i < 256 + 16 + 256 + 16; i += kThreads) sv[Vec::head + i] = __ldg(p.tab + ly.head0 + i);
    const uint32_t bar_full0 = smem_u32(&s_bars[0]), bar_full1 = smem_u32(&s_bars[1]);
    const uint32_t bar_mma[2] = {smem_u32(&s_bars[2]), smem_u32(&s_bars[3])};
    if (tid == 0) { mbar_init(bar_full0, 1); mbar_init(bar_full1, 1); mbar_init(bar_mma[0], 1); mbar_init(bar_mma[1], 1); }
    if (warp == 0) tmem_alloc(smem_u32(&s_tmem_slot), 512);
    fence_barrier_init();
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, s_tmem_slot, 0);
    const uint32_t lane_off = ((uint32_t)(qq * 32) << 16);
    const int col0 = cq * kCW;
    const uint32_t dX[2] = {tmem, tmem + 256}, dACC[2] = {tmem + 128, tmem + 384};

    const int n_tiles = p.pack[5];
    const int32_t* tile_recs = p.pack + 8 + (size_t)p.B * 4;
    const int n_pairs = (n_tiles + 1) / 2;
    const int my_pairs = n_pairs > (int)blockIdx.x ? (n_pairs - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const uint32_t total_mats = (uint32_t)my_pairs * ly.n_seq;
    const uint32_t wbase = smem_u32(smem + kOffRing);
    auto issue_load = [&](uint32_t i) {   // thread 0 only
        const uint32_t bar = (i & 1) ? bar_full1 : bar_full0;
        mbar_expect_tx(bar, kSlot);
        bulk_g2s(wbase + (i & 1) * kSlot, p.image + (size_t)(i % ly.n_seq) * kSlot, kSlot, bar);
    };
    if (tid == 0) {
        if (total_mats > 0) issue_load(0);
        if (total_mats > 1) issue_load(1);
    }
    uint32_t wseq = 0;                 // streamed matrix the next GEMM phase consumes
    uint32_t mma_phase[2] = {0, 0};
    constexpr uint32_t idesc128 = instr_desc(128, 128), idesc16 = instr_desc(128, 16);
    const uint64_t ones_desc = smem_desc(smem_u32(sOnes), 128, 256);

    // D (+)= A[128 x 16 nk] W^T with streamed matrix `ws` (+ bias K-step); commit to the tile's barrier.  One elected lane of warp 0.
    auto gemm = [&](int t, uint32_t ws, uint32_t d, int nk, uint32_t idesc, bool accumulate, bool bias) {
        if (warp == 0) {
            const uint32_t w = __shfl_sync(0xffffffffu, ws, 0);
            if (elect_one()) {
                const uint32_t wb = wbase + (w & 1) * kSlot;
                mbar_wait((w & 1) ? bar_full1 : bar_full0, (w >> 1) & 1);
                tc_fence_after();
                const uint64_t ad = smem_desc(smem_u32(sA(t)), 128, 2048), wd = smem_desc(wb, 128, 2048);
#pragma unroll 8
                for (int j = 0; j < nk; ++j) umma(d, ad + (uint64_t)(j * 16), wd + (uint64_t)(j * 16), idesc, (accumulate || j > 0) ? 1u : 0u);
                if (bias) umma(d, ones_desc, smem_desc(wb + kSlotBias, 128, 256), idesc, 1u);
                umma_commit(bar_mma[t]);
            }
            __syncwarp();
        }
    };
    auto wait_tile = [&](int t) {
        mbar_wait(bar_mma[t], mma_phase[t]); mma_phase[t] ^= 1;
        tc_fence_after();
    };
    // matrix `wseq` has served both tiles: its ring slot is free -> prefetch the matrix two ahead
    auto matrix_done = [&]() {
        if (tid == 0 && wseq + 2 < total_mats) issue_load(wseq + 2);
        ++wseq;
    };
    // (A dedicated issuer warp fed through arrive-only barriers was tried: the issue latency leaves the epilogue warps, but a 17th
    // warp costs a 4-warp register granule — 96 registers, spills in the per-jet path — and the epilogues then wait for the GEMM
    // they used to overlap: 0.455 ms against 0.443 ms at 4096 jets.)
    auto publish = [&]() {   // operand tile / TMEM writes of all threads -> visible to the MMA proxy, then the block barrier
        tc_fence_before();
        fence_proxy_async();
        __syncthreads();
    };
    auto compute_sync = [&]() { __syncthreads(); };

    // ---- one stage of the per-jet path: c = W in for the jets of the CTA (rows g < kMaxJ of an m16 tile).  Warp w < n_warps owns
    // outputs 8 w .. 8 w + 7; on return lane (g, t4) holds outputs 8 w + 2 t4, + 1 of jet g in c[0], c[1].  The weight fragments
    // do not depend on the data: `frag_load` issues all of a stage's loads at once (one L2 latency per stage) and may be called
    // before the barrier that publishes the stage's input.
    constexpr int kMaxKS = (256 + kMaxTXq + kMaxGq) / 16;
    static_assert(kMaxKS % 2 == 0, "stage() walks the k-steps in pairs");
    auto frag_load = [&](const uint2* base, int KS, int n_warps, auto& f) {   // one 16-byte load per lane and pair of k-steps
        constexpr int cap = sizeof(f.b) / sizeof(uint2);
        static_assert(cap % 2 == 0, "fragments travel in pairs of k-steps");
        const uint4* b4 = reinterpret_cast<const uint4*>(base) + (size_t)warp * ((KS + 1) / 2) * 32 + lane;
#pragma unroll
        for (int kk = 0; kk < cap; kk += 2) {
            const uint4 q = (warp < n_warps && kk < KS) ? __ldg(b4 + (kk / 2) * 32) : make_uint4(0u, 0u, 0u, 0u);
            f.b[kk] = make_uint2(q.x, q.y);
            f.b[kk + 1] = make_uint2(q.z, q.w);
        }
    };
    // `lo_from`: first k-step whose input also enters with its low half (the 256 pooled features of fc_global1 / global_0 enter as
    // plain bf16 like every activation of the particle GEMMs; the m16n8k16 rate, one per 8 cycles per scheduler, is what bounds a stage)
    auto stage = [&](const auto& f, int KS, int n_warps, const uint32_t* in_hi, const uint32_t* in_lo, int stride, float (&c)[4], int lo_from = 0) {
        constexpr int cap = sizeof(f.b) / sizeof(uint2);
        const uint2* fb = f.b;
        // four independent accumulation chains (hi / lo x even / odd k-step): a chain of dependent MMAs costs ~20 cycles a link
        float ca[4] = {0.f, 0.f, 0.f, 0.f}, cb[4] = {0.f, 0.f, 0.f, 0.f}, cc[4] = {0.f, 0.f, 0.f, 0.f}, cd[4] = {0.f, 0.f, 0.f, 0.f};
        if (warp < n_warps) {
            const uint32_t* h = in_hi + g * stride + t4;
            const uint32_t* l = in_lo + g * stride + t4;
            const bool on = g < kMaxJ;
#pragma unroll
            for (int kk = 0; kk < cap; kk += 2) {
                if (kk < KS) {
                    mma_bf16(ca, on ? h[8 * kk] : 0u, on ? h[8 * kk + 4] : 0u, fb[kk]);
                    if (kk >= lo_from) mma_bf16(cb, on ? l[8 * kk] : 0u, on ? l[8 * kk + 4] : 0u, fb[kk]);
                }
                if (kk + 1 < KS) {
                    mma_bf16(cc, on ? h[8 * kk + 8] : 0u, on ? h[8 * kk + 12] : 0u, fb[kk + 1]);
                    if (kk + 1 >= lo_from) mma_bf16(cd, on ? l[8 * kk + 8] : 0u, on ? l[8 * kk + 12] : 0u, fb[kk + 1]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) c[i] = (ca[i] + cc[i]) + (cb[i] + cd[i]);
    };
    // pooled sums of both tiles -> [mean | sum] of the jets' input vectors (epic.py:136-143); thread = (jet, column pair)
    auto pool_to_input = [&]() {
        if (tid < kMaxJ * 64) {
            const int j = tid >> 6, cp = tid & 63, t = j >> 1, s = j & 1, c = 2 * cp;
            float s0 = 0.0f, s1 = 0.0f;
            int m = 1;
            if (s < s_rec[t][0]) {
                const int q0 = s_rec[t][2 + 4 * s], nq = s_rec[t][3 + 4 * s];
                m = s_rec[t][4 + 4 * s];
                const float* part = sv + Vec::part + t * 16 * 32 + (c >> 5) * 4 * 32 + (c & 31);   // warps 4 cq + q hold column c of quarter q
                for (int q = q0; q < q0 + nq; ++q) { s0 += part[q * 32]; s1 += part[q * 32 + 1]; }
            }
            const float inv = 1.0f / (float)m;
            uint32_t hi, lo;
            split_pair(s0 * inv, s1 * inv, hi, lo);
            sw[Vec::in1_hi + j * kIn1Stride + cp] = hi; sw[Vec::in1_lo + j * kIn1Stride + cp] = lo;
            split_pair(s0, s1, hi, lo);
            sw[Vec::in1_hi + j * kIn1Stride + 64 + cp] = hi; sw[Vec::in1_lo + j * kIn1Stride + 64 + cp] = lo;
        }
    };
    // lanes (g < kMaxJ) of the warps that own outputs: store a pair of a 128-vector as bf16 hi / lo words
    auto put_pair = [&](int hi_off, int lo_off, int stride, int word, float v0, float v1) {
        uint32_t hi, lo;
        split_pair(v0, v1, hi, lo);
        sw[hi_off + g * stride + word] = hi;
        sw[lo_off + g * stride + word] = lo;
    };

    for (int pi = 0; pi < my_pairs; ++pi) {
        const int pair = (int)blockIdx.x + pi * (int)gridDim.x;
        // ---- the pair's tiles: records, row map (row i of a segment = its i-th live particle), context vectors ---------------
        if (tid < 2 * kRec) {
            const int t = tid / kRec, i = tid % kRec, tile = 2 * pair + t;
            s_rec[t][i] = tile < n_tiles ? __ldg(tile_recs + (size_t)tile * kRec + i) : 0;
        }
        if (tid < 256) s_slot[tid] = -1;
        __syncthreads();
        const bool has_b = s_rec[1][0] > 0;
        if (tid < 8) {
            const int t = tid >> 2, q = tid & 3;
            int sg = -1;
            for (int s = 0; s < s_rec[t][0]; ++s)
                if (q >= s_rec[t][2 + 4 * s] && q < s_rec[t][2 + 4 * s] + s_rec[t][3 + 4 * s]) sg = s;
            s_qseg[t][q] = sg;
        }
        if (warp < kMaxJ) {   // warp j: mask of jet j -> ranks
            const int t = warp >> 1, s = warp & 1;
            if (s < s_rec[t][0]) {
                const int jet = s_rec[t][1 + 4 * s], base = 32 * s_rec[t][2 + 4 * s];
                int before = 0;
                for (int n0 = 0; n0 < p.N; n0 += 32) {
                    const int n = n0 + lane;
                    const bool on = n < p.N && p.mask[(size_t)jet * p.N + n] != 0;
                    const uint32_t bits = __ballot_sync(0xffffffffu, on);
                    if (on) s_slot[t * 128 + base + before + __popc(bits & ((1u << lane) - 1u))] = n;
                    before += __popc(bits);
                }
            }
        } else if (warp < 2 * kMaxJ) {   // warp 4 + j: context vector [time embedding | embedded context] of jet j, zero padded
            const int j = warp - kMaxJ, t = j >> 1, s = j & 1;
            const bool on = s < s_rec[t][0];
            const int jet = on ? s_rec[t][1 + 4 * s] : 0;
            for (int w = lane; w < kMaxTXq / 2; w += 32) {
                const float v0 = (on && 2 * w < TX) ? __ldg(p.temb + (size_t)jet * p.temb_stride + 2 * w) : 0.0f;
                const float v1 = (on && 2 * w + 1 < TX) ? __ldg(p.temb + (size_t)jet * p.temb_stride + 2 * w + 1) : 0.0f;
                uint32_t hi, lo;
                split_pair(v0, v1, hi, lo);
                sw[Vec::in1_hi + j * kIn1Stride + 128 + w] = hi; sw[Vec::in1_lo + j * kIn1Stride + 128 + w] = lo;
                sw[Vec::cx_hi + j * kCxStride + w] = hi; sw[Vec::cx_lo + j * kCxStride + w] = lo;
            }
        }
        compute_sync();
        // ---- per-thread facts of the pair; first operand rows [x_hi, x_lo, onehot(k)]
        int slot[2], seg[2], jetr[2];
        bool live[2];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            slot[t] = s_slot[t * 128 + r];
            live[t] = slot[t] >= 0;
            seg[t] = s_qseg[t][qq];                               // warp-uniform
            jetr[t] = seg[t] >= 0 ? s_rec[t][1 + 4 * seg[t]] : 0;
        }
        if (cq < 2) {
            const int t = cq;
            uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (live[t]) {
                const size_t pidx = (size_t)jetr[t] * p.N + slot[t];
                const float* xr = p.x + pidx * 3;
                const float x0 = xr[0], x1 = xr[1], x2 = xr[2];
                const float h0 = __bfloat162float(__float2bfloat16(x0)), h1 = __bfloat162float(__float2bfloat16(x1)),
                            h2 = __bfloat162float(__float2bfloat16(x2));
                const int kk = p.k[pidx];
                w[0] = pack_bf16(h0, h1); w[1] = pack_bf16(h2, x0 - h0); w[2] = pack_bf16(x1 - h1, x2 - h2);
                const int pos = 6 + kk;   // onehot column
                w[pos >> 1] |= 0x3F80u << (16 * (pos & 1));
            }
            uint8_t* q = sA(t) + (r >> 3) * 2048 + (r & 7) * 16;
            *reinterpret_cast<uint4*>(q) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(q + 128) = make_uint4(w[4], w[5], w[6], w[7]);
        }
        publish();
        // ---- local_0 (one K-step) for both tiles; meanwhile the per-jet time vector of its bias -> bl1 buffer
        gemm(0, wseq, dX[0], 1, idesc128, false, false);
        if (has_b) gemm(1, wseq, dX[1], 1, idesc128, false, false);
        {
            FragRegs<kMaxTXq / 16> f;
            float c[4];
            frag_load(p.frag + ly.f_w0t, ly.KS_t(), 16, f);
            const float2 c0 = __ldg(reinterpret_cast<const float2*>(p.tab + ly.c0 + 8 * warp + 2 * t4));
            stage(f, ly.KS_t(), 16, sw + Vec::in1_hi + 128, sw + Vec::in1_lo + 128, kIn1Stride, c);
            if (g < kMaxJ) {
                const int o = 8 * warp + 2 * t4;
                sv[Vec::bl1 + g * 128 + o] = c[0] + c0.x;
                sv[Vec::bl1 + g * 128 + o + 1] = c[1] + c0.y;
            }
        }
        compute_sync();
        // epilogue of a particle Linear: bias -> leaky-ReLU (-> + skip) -> bf16 operand tile (and fp32 X, pooling sums)
        // kind 0: local_0 (X = lrelu(X + tv0); defines the skip); 1: fc_local1 (A = lrelu(ACC + bl1)); 2: fc_local2 (X = lrelu(X) + skip)
        auto epilogue = [&](int t, int kind, bool last) {
            wait_tile(t);
            const bool warp_live = __any_sync(0xffffffffu, live[t]);
            float v[32];
            if (warp_live) {
                tmem_ld32((kind == 1 ? dACC[t] : dX[t]) + lane_off + col0, v);
                if (kind != 2) {
                    const float* b = sv + Vec::bl1 + (2 * t + seg[t]) * 128 + col0;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 b4 = *reinterpret_cast<const float4*>(b + j);
                        v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                    }
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = lrelu(v[j]);
                if (kind != 1) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = live[t] ? v[j] : 0.0f;   // select: an unused row may hold anything
                    if (skip_on) {
                        if (kind == 0) {
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                *skip_chunk(sSkip(t), r, 4 * cq + c) = make_uint4(pack_f16(v[8 * c], v[8 * c + 1]), pack_f16(v[8 * c + 2], v[8 * c + 3]),
                                                                                  pack_f16(v[8 * c + 4], v[8 * c + 5]), pack_f16(v[8 * c + 6], v[8 * c + 7]));
                        } else {
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const uint4 s4 = *skip_chunk(sSkip(t), r, 4 * cq + c);
                                const uint32_t sk[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&sk[i]));
                                    v[8 * c + 2 * i] += f.x; v[8 * c + 2 * i + 1] += f.y;
                                }
                            }
                        }
                    }
                    tmem_st32(dX[t] + lane_off + col0, v);
                    if (last && p.hidden_out && live[t]) {   // the last local hidden (EPiCWrapper.forward(output_hidden_local=True), epic.py:159-160)
                        float* h = p.hidden_out + ((size_t)jetr[t] * p.N + slot[t]) * kH + col0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(h + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                    }
                }
                store_row(sA(t), r, col0, v);
                if (kind != 1) {   // column sums for the next pooling (unused rows are zero already)
                    warp_halving_sum(v, lane);
                    sv[Vec::part + t * 16 * 32 + warp * 32 + warp_halving_index<32>(lane)] = v[0];
                }
            } else if (kind != 1) {
                sv[Vec::part + t * 16 * 32 + warp * 32 + lane] = 0.0f;
            }
        };
        epilogue(0, 0, false);
        publish();
        gemm(0, wseq + 1, dACC[0], 8, idesc128, false, false);                       // fc_local1 of layer 0, tile A
        if (has_b) epilogue(1, 0, false);
        publish();
        matrix_done();                                                               // local_0 served both tiles
        if (has_b) gemm(1, wseq, dACC[1], 8, idesc128, false, false);
        // ---- EPiC_Projection globals (epic.py:187-190): g0 = lrelu(G0 [mean, sum, ctx]), g1 = lrelu(G1 g0), xg = lrelu(G2 g1)
        {
            FragRegs<kMaxKS> f;
            FragRegs<8> f1, f2;
            float c[4];
            frag_load(p.frag + ly.f_g0, ly.KS_0(), 16, f);     // all three stages' fragments in flight at once: one L2 latency
            frag_load(p.frag + ly.f_g1, 8, 16, f1);
            frag_load(p.frag + ly.f_g2, 8, Gq / 8, f2);
            const int ob = 8 * warp + 2 * t4;                  // ... and the biases this lane will add
            const float2 bias0 = __ldg(reinterpret_cast<const float2*>(p.tab + ly.b_g0 + ob));
            const float2 bias1 = __ldg(reinterpret_cast<const float2*>(p.tab + ly.b_g1 + ob));
            const float2 bias2 = warp < Gq / 8 ? __ldg(reinterpret_cast<const float2*>(p.tab + ly.b_g2 + ob)) : make_float2(0.f, 0.f);
            pool_to_input();
            compute_sync();
            stage(f, ly.KS_0(), 16, sw + Vec::in1_hi, sw + Vec::in1_lo, kIn1Stride, c, 16);
            if (g < kMaxJ) put_pair(Vec::gva_hi, Vec::gva_lo, kGvStride, 4 * warp + t4, lrelu(c[0] + bias0.x), lrelu(c[1] + bias0.y));
            compute_sync();
            stage(f1, 8, 16, sw + Vec::gva_hi, sw + Vec::gva_lo, kGvStride, c);
            if (g < kMaxJ) put_pair(Vec::gvb_hi, Vec::gvb_lo, kGvStride, 4 * warp + t4, lrelu(c[0] + bias1.x), lrelu(c[1] + bias1.y));
            compute_sync();
            stage(f2, 8, Gq / 8, sw + Vec::gvb_hi, sw + Vec::gvb_lo, kGvStride, c);
            if (g < kMaxJ && warp < Gq / 8) {
                const int o = 8 * warp + 2 * t4;
                const float x0 = o < G ? lrelu(c[0] + bias2.x) : 0.0f, x1 = o + 1 < G ? lrelu(c[1] + bias2.y) : 0.0f;
                sv[Vec::xg + g * kMaxGq + o] = x0; sv[Vec::xg + g * kMaxGq + o + 1] = x1;
                sv[Vec::skg + g * kMaxGq + o] = skip_on ? x0 : 0.0f; sv[Vec::skg + g * kMaxGq + o + 1] = skip_on ? x1 : 0.0f;
                put_pair(Vec::in1_hi, Vec::in1_lo, kIn1Stride, 128 + TXq / 2 + 4 * warp + t4, x0, x1);
            }
            compute_sync();
        }
        // ---- EPiC layers (epic.py:217-241, 152-155)
        for (int l = 0; l < L; ++l) {
            const float* tl = p.tab + ly.layer0 + (size_t)l * ly.layer_stride;
            const uint2* fl = p.frag + ly.f_layer0 + (size_t)l * ly.f_layer_stride;
            {   // per-jet path: fc_global1 -> fc_global2 (+ residual) -> the per-jet part of fc_local1
                FragRegs<kMaxKS> f;
                FragRegs<8> f2;
                FragRegs<(kMaxTXq + kMaxGq) / 16> f3;
                float c[4];
                frag_load(fl + ly.fo_wg1, ly.KS_1(), 16, f);   // all three stages' fragments in flight at once: one L2 latency
                frag_load(fl + ly.fo_wg2, 8, Gq / 8, f2);
                frag_load(fl + ly.fo_wl1g, ly.KS_2(), 16, f3);
                // ... and the biases this lane will add (a load at the end of a stage would put an L2 latency on the chain)
                const int ob = 8 * warp + 2 * t4;
                const float2 bias1 = __ldg(reinterpret_cast<const float2*>(tl + ly.o_blg1 + ob));
                const float2 bias2 = warp < Gq / 8 ? __ldg(reinterpret_cast<const float2*>(tl + ly.o_blg2 + ob)) : make_float2(0.f, 0.f);
                const float2 bias3 = __ldg(reinterpret_cast<const float2*>(tl + ly.o_bl1 + ob));
                if (l > 0) {
                    pool_to_input();
                    compute_sync();
                }
                stage(f, ly.KS_1(), 16, sw + Vec::in1_hi, sw + Vec::in1_lo, kIn1Stride, c, 16);
                if (g < kMaxJ) put_pair(Vec::gva_hi, Vec::gva_lo, kGvStride, 4 * warp + t4, lrelu(c[0] + bias1.x), lrelu(c[1] + bias1.y));
                compute_sync();
                stage(f2, 8, Gq / 8, sw + Vec::gva_hi, sw + Vec::gva_lo, kGvStride, c);
                if (g < kMaxJ && warp < Gq / 8) {
                    const int o = 8 * warp + 2 * t4;
                    float* xg = sv + Vec::xg + g * kMaxGq + o;
                    const float* sk = sv + Vec::skg + g * kMaxGq + o;
                    const float m0 = o < G ? lrelu(c[0] + bias2.x + xg[0]) : 0.0f, m1 = o + 1 < G ? lrelu(c[1] + bias2.y + xg[1]) : 0.0f;
                    put_pair(Vec::cx_hi, Vec::cx_lo, kCxStride, TXq / 2 + 4 * warp + t4, m0, m1);              // fc_local1 sees the layer's own output
                    xg[0] = m0 + sk[0]; xg[1] = m1 + sk[1];                                                    // the next layer the skipped one (epic.py:155)
                    put_pair(Vec::in1_hi, Vec::in1_lo, kIn1Stride, 128 + TXq / 2 + 4 * warp + t4, xg[0], xg[1]);
                }
                compute_sync();
                stage(f3, ly.KS_2(), 16, sw + Vec::cx_hi, sw + Vec::cx_lo, kCxStride, c);
                if (g < kMaxJ) {
                    const int o = 8 * warp + 2 * t4;
                    sv[Vec::bl1 + g * 128 + o] = c[0] + bias3.x;
                    sv[Vec::bl1 + g * 128 + o + 1] = c[1] + bias3.y;
                }
                compute_sync();
            }
            const bool last = l == L - 1;
            epilogue(0, 1, false);
            publish();
            gemm(0, wseq + 1, dX[0], 8, idesc128, true, true);                      // fc_local2 accumulates onto X
            if (has_b) epilogue(1, 1, false);
            publish();
            matrix_done();                                                           // fc_local1 served both tiles
            if (has_b) gemm(1, wseq, dX[1], 8, idesc128, true, true);
            epilogue(0, 2, last);
            publish();
            gemm(0, wseq + 1, dACC[0], 8, last ? idesc16 : idesc128, false, last);  // next fc_local1, or the output layer
            if (has_b) epilogue(1, 2, last);
            publish();
            matrix_done();                                                           // fc_local2 served both tiles
            if (has_b) gemm(1, wseq, dACC[1], 8, last ? idesc16 : idesc128, false, last);
        }
        // ---- output layer + discrete head (epic.py:158-162, mbm.py:105-113) for the live particles: the rows of tile A are served by
        // the threads of column slice 0, those of tile B by slice 1, side by side
        wait_tile(0);
        if (has_b) wait_tile(1);
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            if (t == 1 && !has_b) continue;
            if (cq == t) {   // whole warps: tcgen05.ld is warp-collective
                float v[32];
                tmem_ld32(dACC[t] + lane_off, v);
                if (live[t]) {
                    const size_t pidx = (size_t)jetr[t] * p.N + slot[t];
#pragma unroll
                    for (int c = 0; c < 3; ++c) p.v_out[pidx * 3 + c] = v[c];
                    const float* hd = sv + Vec::head;
                    float z1[16], lg[8];
#pragma unroll
                    for (int o = 0; o < 16; ++o) {   // head Linear 0 + SELU (rows >= Sh are zero in the table and unused)
                        float a = hd[256 + o];
#pragma unroll
                        for (int s = 0; s < 8; ++s) a = fmaf(hd[o * 16 + s], v[3 + s], a);
                        z1[o] = selu(a);
                    }
#pragma unroll
                    for (int o = 0; o < 8; ++o) {
                        float a = hd[256 + 16 + 256 + o];
#pragma unroll
                        for (int s = 0; s < 16; ++s) a = fmaf(hd[256 + 16 + o * 16 + s], z1[s], a);
                        lg[o] = Sh ? a : v[3 + o];
                    }
#pragma unroll
                    for (int o = 0; o < 8; ++o)
                        if (o < S) p.logits_out[pidx * S + o] = lg[o];
                }
            }
        }
        tc_fence_before();
        compute_sync();
        matrix_done();   // output layer served both tiles
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

inline uint32_t host_pack_bf16(float lo, float hi) {
    const __nv_bfloat16 a = __float2bfloat16(lo), b = __float2bfloat16(hi);
    return (uint32_t)(*reinterpret_cast<const uint16_t*>(&a)) | ((uint32_t)(*reinterpret_cast<const uint16_t*>(&b)) << 16);
}
// B fragments of y = W x for mma.sync m16n8k16 (col-major B): warp w owns outputs 8 w .. 8 w + 7; entry ((w KS + kk) 32 + lane) =
// {W[n][16 kk + 2 t, + 1], W[n][16 kk + 2 t + 8, + 9]} with n = 8 w + lane / 4, t = lane % 4.  `w(n, k)` returns 0 outside the matrix.
template <typename F>
void put_frag(std::vector<uint2>& img, int base, int n_out, int ks, F w) {
    for (int wp = 0; wp < n_out / 8; ++wp)
        for (int kk = 0; kk < ks; ++kk)
            for (int lane = 0; lane < 32; ++lane) {
                const int n = 8 * wp + lane / 4, k0 = 16 * kk + 2 * (lane % 4);
                // k-steps travel in pairs: lane's entries of k-steps 2 i and 2 i + 1 are adjacent (one 16-byte load)
                img[(size_t)base + (((size_t)wp * ((ks + 1) / 2) + kk / 2) * 32 + lane) * 2 + (kk & 1)] =
                    make_uint2(host_pack_bf16(w(n, k0), w(n, k0 + 1)), host_pack_bf16(w(n, k0 + 8), w(n, k0 + 9)));
            }
}

}  // namespace

struct WideImage {
    void* image = nullptr;
    float* tab = nullptr;
    uint2* frag = nullptr;
    WideLayout lay;
};

bool wide_supported(const MmbEpicDims* d, int N) {
    return d->dim_hidden_local == kH && d->dim_hidden_glob >= 1 && d->dim_hidden_glob <= kMaxGq && d->dim_time_emb >= 1 && d->dim_context >= 0 &&
           d->dim_time_emb + d->dim_context <= kMaxTXq && d->num_blocks >= 1 && d->num_blocks <= kMaxL &&
           d->dim_continuous == 3 && d->vocab_size >= 1 && d->vocab_size <= 8 && d->disc_head_hidden >= 0 && d->disc_head_hidden <= 16 &&
           N >= 1 && N <= 128;
}

void wide_free_image(EpicModel* m) {
    WideImage* w = static_cast<WideImage*>(m->wide);
    if (!w) return;
    if (w->image) cudaFree(w->image);
    if (w->tab) cudaFree(w->tab);
    if (w->frag) cudaFree(w->frag);
    delete w;
    m->wide = nullptr;
}

int wide_build_image(EpicModel* m, const float* W) {
    const MmbEpicDims& d = m->dims;
    const MmbEpicLayout& Lo = m->layout;
    const WideLayout ly = make_layout(d);
    const int T = d.dim_time_emb, X = d.dim_context, TX = T + X, C = d.dim_cont_emb, D = d.dim_disc_emb, G = d.dim_hidden_glob, L = d.num_blocks,
              S = d.vocab_size, Sh = d.disc_head_hidden, Dc = d.dim_continuous, H = kH, TXq = ly.TXq;
    const int K0 = T + C + D;
    std::vector<__nv_bfloat16> img((size_t)ly.n_seq * kSlot / 2, __float2bfloat16(0.0f));
    std::vector<float> tab((size_t)ly.tab_floats, 0.0f);
    std::vector<uint2> frag((size_t)ly.frag_elems, make_uint2(0u, 0u));
    // local_0 with the embeddings folded in: operand columns [x_hi (3) | x_lo (3) | onehot (S)]; its time columns act on the
    // jet's context vector (whose first T entries are the time embedding)
    for (int o = 0; o < H; ++o) {
        const float* w0 = W + Lo.local0_w + (size_t)o * K0;
        for (int j = 0; j < Dc; ++j) {
            double acc = 0;
            for (int c = 0; c < C; ++c) acc += (double)w0[T + c] * W[Lo.emb_cont_w + (size_t)c * Dc + j];
            slot_put_weight(img, 0, o, j, acc);
            slot_put_weight(img, 0, o, Dc + j, acc);
        }
        for (int s = 0; s < S; ++s) {
            double acc = 0;
            for (int dd = 0; dd < D; ++dd) acc += (double)w0[T + C + dd] * W[Lo.emb_disc + (size_t)s * D + dd];
            slot_put_weight(img, 0, o, 2 * Dc + s, acc);
        }
        double c0 = W[Lo.local0_b + o];
        for (int c = 0; c < C; ++c) c0 += (double)w0[T + c] * W[Lo.emb_cont_b + c];
        tab[ly.c0 + o] = (float)c0;
        tab[ly.b_g0 + o] = W[Lo.global0_b + o];
        tab[ly.b_g1 + o] = W[Lo.global1_b + o];
    }
    put_frag(frag, ly.f_w0t, 128, ly.KS_t(), [&](int n, int k) { return k < T ? W[Lo.local0_w + (size_t)n * K0 + k] : 0.0f; });
    // projection globals: global_0 [H][mean | sum | ctx], global_1 [H][H], global_2 [G][H]
    put_frag(frag, ly.f_g0, 128, ly.KS_0(), [&](int n, int k) { return k < 2 * H + TX ? W[Lo.global0_w + (size_t)n * (2 * H + TX) + k] : 0.0f; });
    put_frag(frag, ly.f_g1, 128, 8, [&](int n, int k) { return W[Lo.global1_w + (size_t)n * H + k]; });
    put_frag(frag, ly.f_g2, ly.Gq, 8, [&](int n, int k) { return n < G ? W[Lo.global2_w + (size_t)n * H + k] : 0.0f; });
    for (int o = 0; o < G; ++o) tab[ly.b_g2 + o] = W[Lo.global2_b + o];
    for (int l = 0; l < L; ++l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        float* tl = tab.data() + ly.layer0 + (size_t)l * ly.layer_stride;
        const int fl = ly.f_layer0 + l * ly.f_layer_stride;
        const int Kg = 2 * H + G + TX, Kl = H + G + TX;
        // fc_global1: reference columns [mean | sum | xg | ctx] -> input layout [mean | sum | ctx (TXq) | xg (Gq)]
        put_frag(frag, fl + ly.fo_wg1, 128, ly.KS_1(), [&](int n, int k) {
            const float* g1 = Wl + Lo.l_g1_w + (size_t)n * Kg;
            if (k < 2 * H) return g1[k];
            if (k < 2 * H + TXq) return k - 2 * H < TX ? g1[2 * H + G + (k - 2 * H)] : 0.0f;
            return k - 2 * H - TXq < G ? g1[2 * H + (k - 2 * H - TXq)] : 0.0f;
        });
        put_frag(frag, fl + ly.fo_wg2, ly.Gq, 8, [&](int n, int k) { return n < G ? Wl[Lo.l_g2_w + (size_t)n * H + k] : 0.0f; });
        // fc_local1 [local H | xg | ctx]: the local part streams as matrix 1 + 2l, the per-jet part acts on [ctx (TXq) | xm (Gq)]
        put_frag(frag, fl + ly.fo_wl1g, 128, ly.KS_2(), [&](int n, int k) {
            const float* l1 = Wl + Lo.l_l1_w + (size_t)n * Kl;
            if (k < TXq) return k < TX ? l1[H + G + k] : 0.0f;
            return k - TXq < G ? l1[H + (k - TXq)] : 0.0f;
        });
        for (int o = 0; o < H; ++o) {
            tl[ly.o_blg1 + o] = Wl[Lo.l_g1_b + o];
            tl[ly.o_bl1 + o] = Wl[Lo.l_l1_b + o];
            for (int k = 0; k < H; ++k) slot_put_weight(img, 1 + 2 * l, o, k, Wl[Lo.l_l1_w + (size_t)o * Kl + k]);
            for (int k = 0; k < H; ++k) slot_put_weight(img, 2 + 2 * l, o, k, Wl[Lo.l_l2_w + (size_t)o * H + k]);
            slot_put_bias(img, 2 + 2 * l, o, Wl[Lo.l_l2_b + o]);
        }
        for (int o = 0; o < G; ++o) tl[ly.o_blg2 + o] = Wl[Lo.l_g2_b + o];
    }
    for (int o = 0; o < Dc + S; ++o) {
        for (int k = 0; k < H; ++k) slot_put_weight(img, 1 + 2 * L, o, k, W[Lo.out_w + (size_t)o * H + k]);
        slot_put_bias(img, 1 + 2 * L, o, W[Lo.out_b + o]);
    }
    if (Sh) {   // discrete head; a padded slot's logits are head(0) (the reference masks before the head, mbm.py:105-111)
        std::vector<double> z1(Sh);
        for (int o = 0; o < Sh; ++o) {
            for (int s = 0; s < S; ++s) tab[ly.head0 + o * 16 + s] = W[Lo.head0_w + (size_t)o * S + s];
            tab[ly.b_head0 + o] = W[Lo.head0_b + o];
            const double a = W[Lo.head0_b + o];
            z1[o] = 1.0507009873554804934193349852946 * (a > 0 ? a : 1.6732632423543772848170429916717 * (exp(a) - 1.0));
        }
        for (int o = 0; o < S; ++o) {
            double acc = W[Lo.head2_b + o];
            for (int s = 0; s < Sh; ++s) {
                tab[ly.head2 + o * 16 + s] = W[Lo.head2_w + (size_t)o * Sh + s];
                acc += (double)W[Lo.head2_w + (size_t)o * Sh + s] * z1[s];
            }
            tab[ly.b_head2 + o] = W[Lo.head2_b + o];
            tab[ly.dead_logits + o] = (float)acc;
        }
    }
    WideImage* w = new WideImage();
    w->lay = ly;
    m->wide = w;
    int rc = cuda_ok(cudaMalloc(&w->image, img.size() * 2), "cudaMalloc wide image");
    if (!rc) rc = cuda_ok(cudaMalloc(&w->tab, tab.size() * 4), "cudaMalloc wide table");
    if (!rc) rc = cuda_ok(cudaMalloc(&w->frag, frag.size() * sizeof(uint2)), "cudaMalloc wide fragments");
    if (!rc) rc = cuda_ok(cudaMemcpy(w->image, img.data(), img.size() * 2, cudaMemcpyHostToDevice), "wide image upload");
    if (!rc) rc = cuda_ok(cudaMemcpy(w->tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice), "wide table upload");
    if (!rc) rc = cuda_ok(cudaMemcpy(w->frag, frag.data(), frag.size() * sizeof(uint2), cudaMemcpyHostToDevice), "wide fragments upload");
    if (rc) wide_free_image(m);
    return rc;
}

int launch_epic_forward_wide(const EpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask, const float* temb, int temb_stride,
                             int B, int N, float* v_out, float* logits_out, float* hidden_out, cudaStream_t stream) {
    const WideImage* w = static_cast<const WideImage*>(m->wide);
    if (!w) return fail(MMB_EUNSUPPORTED, "wide EPiC trunk: no operand image for this model");
    if (B == 0 || N == 0) return MMB_OK;
    if (N > 128) return fail(MMB_EUNSUPPORTED, "wide EPiC trunk handles up to 128 particle slots per jet (got %d)", N);
    if (B >= (1 << 20)) return fail(MMB_EUNSUPPORTED, "wide EPiC trunk: at most 2^20 - 1 jets per call");
    // pre-pass scratch (jet lists, tile records): a stream-ordered allocation, so concurrent evaluations on different streams of
    // one model handle never share it and nothing synchronises (the pool reuses the block from call to call)
    int32_t* pack = nullptr;
    if (int rc = cuda_ok(cudaMallocAsync(reinterpret_cast<void**>(&pack), pack_ints(B) * sizeof(int32_t), stream), "wide pre-pass scratch")) return rc;
    WideParams p{};
    p.image = static_cast<const uint8_t*>(w->image); p.tab = w->tab; p.frag = w->frag; p.lay = w->lay; p.pack = pack;
    p.x = x; p.k = k; p.mask = mask; p.temb = temb; p.temb_stride = temb_stride; p.B = B; p.N = N;
    p.v_out = v_out; p.logits_out = logits_out; p.hidden_out = hidden_out;
    int rc = cuda_ok(cudaMemsetAsync(pack, 0, 8 * sizeof(int32_t), stream), "wide pre-pass counters");
    if (!rc) {
        wide_pack_kernel<<<(B + 7) / 8, 256, 0, stream>>>(mask, B, N, w->lay.S, w->tab + w->lay.dead_logits, v_out, logits_out, hidden_out, pack);
        wide_tiles_kernel<<<(B + 255) / 256, 256, 0, stream>>>(pack, B);
        rc = cuda_ok(cudaGetLastError(), "wide pre-pass launch");
    }
    if (!rc) rc = cuda_ok(cudaFuncSetAttribute(epic_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes), "wide smem attribute");
    if (!rc) {
        const int pairs = (B + 1) / 2;   // upper bound of the tile pairs (the kernel reads the count the pre-pass left)
        const int grid = pairs < m->sm_count ? pairs : m->sm_count;
        epic_wide_kernel<<<grid, kThreads, kSmemBytes, stream>>>(p);
        rc = cuda_ok(cudaGetLastError(), "epic_wide launch");
    }
    cudaFreeAsync(pack, stream);   // ordered after the kernel on this stream
    return rc;
}

}  // namespace mmb
