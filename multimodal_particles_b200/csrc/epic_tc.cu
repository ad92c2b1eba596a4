// epic_tc.cu — the EPiC network + hybrid update on 5th-gen tensor cores (tcgen05 / TMEM), sm_100a.
//
// Shape of the problem: the default EPiC (hidden 16) is eight tiny per-particle GEMMs per solver
// step, K = N = 16, separated by element-wise work and two masked poolings — a strictly serial
// chain per jet, 99 steps long.  HBM is irrelevant once the loop is fused (state in registers for
// the whole generation); what bounds it is issue slots and the latency of the chain.  Design:
//
//   * one jet = one UMMA tile: M = 128 rows = the (padded) particles of the jet, thread r of a
//     128-thread group owns particle r, its TMEM lane r and its row of the A operand;
//   * every per-particle Linear is ONE tcgen05.mma (M128 x N16 x K16, bf16 operands from shared
//     memory, fp32 accumulator in TMEM); weights sit in shared memory for the whole kernel in the
//     canonical no-swizzle K-major layout; the epilogue (bias, leaky-ReLU, residual, mask, skip)
//     runs on the accumulator row pulled back with tcgen05.ld and writes the next A operand as bf16;
//   * algebraic folds keep K at 16: W0·[temb, A x + a, E[k]] = (time vector) + (W0c A) x + (W0d E)[k]
//     so the first layer's A row is [x_hi, x_lo, onehot(k)] (x split in two bf16 for 16-bit
//     mantissa); the global vector and the time embedding enter the local layers as a per-jet fp32
//     bias computed once per layer, not as 32 more K columns;
//   * masked sum pooling is a GEMM too: ones[128 x 128] · XL[128 x 16] — the activation tile just
//     written as the next A operand is re-read as an MN-major B operand (K = particles), eight
//     K-steps into a second TMEM accumulator, issued together with the next layer's GEMM.  Every
//     TMEM lane then holds all 16 column sums, so the warp that runs the tiny global MLP reads
//     them with one tcgen05.ld — no shuffles, no shared-memory reduction;
//   * four jets per CTA (512 threads, 64 registers) share one copy of the weights; two CTAs per SM interleave
//     eight chains to hide the MMA -> commit -> mbarrier -> tcgen05.ld round trips;
//   * one warp per jet is "special": an elected lane issues the jet's MMAs and the warp runs the per-jet global MLP.
//     Everything a tcgen05.mma consumes (descriptors, TMEM addresses) derives from broadcast, provably warp-uniform values,
//     otherwise the compiler wraps every MMA in an elect / R2UR.BROADCAST loop;
//   * generation only: a jet's rows are rotated by (global jet index & 3) quarters of the tile, so the live quarters of the
//     four jets of a CTA sit on four different SM sub-partitions; warps whose 32 particles are all dead skip every epilogue
//     (their A rows stay zero, their pooling K-steps are not issued); the special role goes to the warp of the last quarter,
//     and when that warp has no live particle it runs its own copy of the step loop with no per-particle state alive.
//
// Numerics: bf16 operands, fp32 accumulate, fp32 residual stream / biases / global MLP / update.
// Not bit-comparable with the fp32 path; tests/test_gpu_tc.py states the tolerance.
//
// Reference semantics: SURVEY.md §A.2 (mp/models/architectures/epic.py:136-241, utils.py:112-172,
// mp/models/generative/multimodal_bridge_matching.py:90-113,199-216, bridges.py:38-45,106-132,179-201).
#include <cuda_bf16.h>

#include <type_traits>

#include <vector>

#include "mmb_device.cuh"
#include "mmb_internal.h"
#include "tcgen05.cuh"

namespace mmb {
namespace {

constexpr int kH = 16;      // hidden width this path is built for
constexpr int kGP = 32;     // global width, padded
constexpr int kJPC = 4;     // jets per CTA (512 threads); two CTAs per SM -> 8 jets in flight
constexpr int kTmemPerJet = 64;  // columns: main 16 | pool 16 | skip 16 | spare (allocation must be a power of two)
constexpr int kRows = 128;  // UMMA M
constexpr int kMaxL = 4;
constexpr int kMaxT = 32;
constexpr int kS16 = 20, kS32 = 36;   // padded row strides (floats) of the global-MLP matrices with 16 / 32 inputs

// ---- image layout (host builds, kernel copies to shared memory) --------------------------------
// bf16 region: n_bops matrices of [16 out][16 k] in UMMA canonical K-major no-swizzle layout
//   (core matrix = 8 rows x 16 B; k-chunks 128 B apart (LBO), 8-row groups 256 B apart (SBO)).
// fp32 region: vectors, [t][o] time matrices (o fastest), and the matrices of the per-jet global MLP as [o][k] rows with k
// contiguous and a padded row stride (kS16 / kS32 floats): a lane reads its 8-16 weights with 128-bit loads, conflict-free.
struct TcLayout {
    int L, G, T, Sh, skip, n_bops;
    // float offsets
    int b0, c0, w0t, g0ms, g0t, g0b, g1, g1b, g2, g2b, layer0, layer_stride;
    int l_g1ms, l_g1g, l_g1t, l_g1b, l_g2, l_g2b, l_l1g, l_l1t, l_l1b, l_l2b;  // within a layer
    int bout, bh0, bh2, n_floats;
    __host__ __device__ int bop_local0() const { return 0; }
    __host__ __device__ int bop_l1(int l) const { return 1 + 2 * l; }
    __host__ __device__ int bop_l2(int l) const { return 2 + 2 * l; }
    __host__ __device__ int bop_out() const { return 1 + 2 * L; }
    __host__ __device__ int bop_h2() const { return 3 + 2 * L; }
    // bias operands ([o][0] = hi, [o][1] = lo as bf16): consumed as one more K-step against a mask/ones A tile
    // every weight operand w has a low-order companion at w + n_weights(): W = hi + lo with both halves
    // bf16, issued as two K-steps, so the weights enter with ~16 mantissa bits (the activations stay bf16)
    __host__ __device__ int n_weights() const { return 4 + 2 * L; }
    __host__ __device__ int bop_bias_l2(int l) const { return 8 + 4 * L + l; }
    __host__ __device__ int bop_bias_out() const { return 8 + 5 * L; }
    __host__ __device__ int bop_bias_h0() const { return 9 + 5 * L; }
    __host__ __device__ int bop_bias_h2() const { return 10 + 5 * L; }
};

TcLayout make_layout(const MmbEpicDims& d) {
    TcLayout t{};
    t.L = d.num_blocks; t.G = d.dim_hidden_glob; t.T = d.dim_time_emb; t.Sh = d.disc_head_hidden; t.skip = d.skip_connection;
    t.n_bops = 11 + 5 * t.L;
    int o = 0;
    auto take = [&](int n) { int r = o; o += n; return r; };
    t.b0 = take(16); t.c0 = take(16); t.w0t = take(t.T * 16);
    t.g0ms = take(16 * kS32); t.g0t = take(t.T * 16); t.g0b = take(16);   // [o][mean 16 | sum 16]
    t.g1 = take(16 * kS16); t.g1b = take(16);
    t.g2 = take(kGP * kS16); t.g2b = take(kGP);
    t.layer0 = o;
    {
        int p = 0;
        auto tk = [&](int n) { int r = p; p += n; return r; };
        t.l_g1ms = tk(16 * kS32); t.l_g1g = tk(16 * kS32); t.l_g1t = tk(t.T * 16); t.l_g1b = tk(16);
        t.l_g2 = tk(kGP * kS16); t.l_g2b = tk(kGP);
        t.l_l1g = tk(16 * kS32); t.l_l1t = tk(t.T * 16); t.l_l1b = tk(16); t.l_l2b = tk(16);
        t.layer_stride = p;
    }
    o += t.layer_stride * t.L;
    t.bout = take(16); t.bh0 = take(16); t.bh2 = take(16);
    t.n_floats = (o + 3) & ~3;
    return t;
}

// element (row, k) of a [16 x 16] K-major operand -> index in bf16 units
inline int bop_index(int row, int k) { return (row / 8) * 128 + (k / 8) * 64 + (row % 8) * 8 + (k % 8); }

// named_bar(id, 128) with the thread count as an immediate (named_bar passes it in a register)
__device__ __forceinline__ void group_bar(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

// The pooling GEMM: up to eight K-steps (B descriptor advances by 512 B = 32 address units per step) into one accumulator.
// All descriptors are formed before the first MMA so their moves to uniform registers can overlap; K-steps whose bit in
// `live` is clear are skipped (their rows are all zero); the first issued step overwrites, the rest accumulate.
__device__ __forceinline__ void umma_pool8(uint32_t d_tmem, uint64_t adesc, uint64_t adesc_hi, uint64_t bdesc0, uint32_t idesc, uint32_t live) {
    if (live == 0u) live = 1u;   // nothing live: one step over zero rows still defines the accumulator
    const uint32_t first = live & (0u - live);   // lowest set bit: the step that does not accumulate
    asm volatile(
        "{\n\t"
        ".reg .pred e0, e1, e2, e3, e4, e5, e6, e7, a0, a1, a2, a3, a4, a5, a6, a7;\n\t"
        ".reg .b64 b1, b2, b3, b4, b5, b6, b7;\n\t"
        ".reg .b32 t;\n\t"
        "add.s64 b1, %2, 32;\n\t add.s64 b2, %2, 64;\n\t add.s64 b3, %2, 96;\n\t add.s64 b4, %2, 128;\n\t"
        "add.s64 b5, %2, 160;\n\t add.s64 b6, %2, 192;\n\t add.s64 b7, %2, 224;\n\t"
        "and.b32 t, %4, 1;\n\t setp.ne.b32 e0, t, 0;\n\t and.b32 t, %4, 2;\n\t setp.ne.b32 e1, t, 0;\n\t"
        "and.b32 t, %4, 4;\n\t setp.ne.b32 e2, t, 0;\n\t and.b32 t, %4, 8;\n\t setp.ne.b32 e3, t, 0;\n\t"
        "and.b32 t, %4, 16;\n\t setp.ne.b32 e4, t, 0;\n\t and.b32 t, %4, 32;\n\t setp.ne.b32 e5, t, 0;\n\t"
        "and.b32 t, %4, 64;\n\t setp.ne.b32 e6, t, 0;\n\t and.b32 t, %4, 128;\n\t setp.ne.b32 e7, t, 0;\n\t"
        "setp.ne.b32 a0, %5, 1;\n\t setp.ne.b32 a1, %5, 2;\n\t setp.ne.b32 a2, %5, 4;\n\t setp.ne.b32 a3, %5, 8;\n\t"
        "setp.ne.b32 a4, %5, 16;\n\t setp.ne.b32 a5, %5, 32;\n\t setp.ne.b32 a6, %5, 64;\n\t setp.ne.b32 a7, %5, 128;\n\t"
        "@e0 tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, a0;\n\t"
        "@e1 tcgen05.mma.cta_group::1.kind::f16 [%0], %1, b1, %3, a1;\n\t"
        "@e2 tcgen05.mma.cta_group::1.kind::f16 [%0], %1, b2, %3, a2;\n\t"
        "@e3 tcgen05.mma.cta_group::1.kind::f16 [%0], %1, b3, %3, a3;\n\t"
        "@e4 tcgen05.mma.cta_group::1.kind::f16 [%0], %6, b4, %3, a4;\n\t"
        "@e5 tcgen05.mma.cta_group::1.kind::f16 [%0], %6, b5, %3, a5;\n\t"
        "@e6 tcgen05.mma.cta_group::1.kind::f16 [%0], %6, b6, %3, a6;\n\t"
        "@e7 tcgen05.mma.cta_group::1.kind::f16 [%0], %6, b7, %3, a7;\n\t"
        "}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc0), "r"(idesc), "r"(live), "r"(first), "l"(adesc_hi) : "memory");
}

// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// this thread's 16-wide row -> its slot of the A operand (two 16-byte chunks, K-major canonical)
__device__ __forceinline__ void store_a_row(uint8_t* abuf, int row, const float (&v)[16]) {
    uint8_t* p = abuf + (row >> 3) * 256 + (row & 7) * 16;
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    *reinterpret_cast<uint4*>(p + 128) = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
}

// same, rows of dead particles written as zeros (the mask multiply of epic.py:191,241 at pack time)
__device__ __forceinline__ void store_a_row_masked(uint8_t* abuf, int row, const float (&v)[16], bool live) {
    uint8_t* p = abuf + (row >> 3) * 256 + (row & 7) * 16;
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = live ? pack_bf16(v[2 * i], v[2 * i + 1]) : 0u;
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    *reinterpret_cast<uint4*>(p + 128) = make_uint4(w[4], w[5], w[6], w[7]);
}

// 16 floats from 16-byte aligned shared memory
__device__ __forceinline__ void lds16(const float* p, float (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 q = reinterpret_cast<const float4*>(p)[i];
        v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    }
}

// park 16 fp32 values in this thread's TMEM lane (the trunk's skip connection lives there between layers)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                   "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
                   "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
                   "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
                 : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// init + sum_{k<K} w[k * wstride] * x(k) with four independent accumulators: the serial per-jet global MLP is a chain of such
// dots on one warp, and a single accumulator makes every one of them K dependent FMAs long
// init + sum_k w[k] x[k] over K contiguous floats (K % 4 == 0); w and x 16-byte aligned shared memory: 128-bit loads
template <int K>
__device__ __forceinline__ float dotv(float init, const float* w, const float* x) {
    float a0 = init, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
    for (int k = 0; k < K; k += 4) {
        const float4 a = *reinterpret_cast<const float4*>(w + k), b = *reinterpret_cast<const float4*>(x + k);
        a0 = fmaf(a.x, b.x, a0); a1 = fmaf(a.y, b.y, a1); a2 = fmaf(a.z, b.z, a2); a3 = fmaf(a.w, b.w, a3);
    }
    return (a0 + a1) + (a2 + a3);
}
// the same with x in registers, scaled by sc
__device__ __forceinline__ float dotr16(float init, const float* w, const float (&x)[16], float sc) {
    float a0 = init, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
    for (int k = 0; k < 16; k += 4) {
        const float4 a = *reinterpret_cast<const float4*>(w + k);
        a0 = fmaf(a.x, x[k] * sc, a0); a1 = fmaf(a.y, x[k + 1] * sc, a1); a2 = fmaf(a.z, x[k + 2] * sc, a2); a3 = fmaf(a.w, x[k + 3] * sc, a3);
    }
    return (a0 + a1) + (a2 + a3);
}
template <int K, typename XF>
__device__ __forceinline__ float dot4(float init, const float* w, int wstride, XF x) {
    float a0 = init, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
    for (int k = 0; k < K; k += 4) {
        a0 = fmaf(w[(k + 0) * wstride], x(k + 0), a0);
        a1 = fmaf(w[(k + 1) * wstride], x(k + 1), a1);
        a2 = fmaf(w[(k + 2) * wstride], x(k + 2), a2);
        a3 = fmaf(w[(k + 3) * wstride], x(k + 3), a3);
    }
    return (a0 + a1) + (a2 + a3);
}
// out = lrelu(a [+ b]) on 16 values with packed fp32 pair instructions (one FADD2 + one FMUL2 + two FMNMX per pair)
__device__ __forceinline__ void lrelu16(float (&out)[16], const float (&a)[16]) {
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
        float t0, t1;
        fmul2(t0, t1, a[i], a[i + 1], 0.01f, 0.01f);
        out[i] = fmaxf(a[i], t0);
        out[i + 1] = fmaxf(a[i + 1], t1);
    }
}
__device__ __forceinline__ void lrelu16_sum(float (&out)[16], const float (&a)[16], const float (&b)[16]) {
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
        float s0, s1, t0, t1;
        fadd2(s0, s1, a[i], a[i + 1], b[i], b[i + 1]);
        fmul2(t0, t1, s0, s1, 0.01f, 0.01f);
        out[i] = fmaxf(s0, t0);
        out[i + 1] = fmaxf(s1, t1);
    }
}
__device__ __forceinline__ float selu_fast(float a) {
    const float scale = 1.0507009873554804934193349852946f;
    const float alpha_scale = 1.0507009873554804934193349852946f * 1.6732632423543772848170429916717f;
    return a > 0.0f ? scale * a : alpha_scale * (__expf(a) - 1.0f);
}

struct TcParams {
    const uint8_t* image;  // [bf16 bops][fp32 region]
    TcLayout lay;
    // state / inputs
    float* x;              // GENERATE: in/out [B,N,Dc]; forward: in
    uint8_t* k;            // GENERATE: in/out [B,N];    forward: in
    const uint8_t* mask;
    const float* temb;     // forward: [B or 1][T] with stride; generate: table temb [n_steps][T]
    int temb_stride;
    const float* step_tab; // generate: [n_steps][4] (bc, cc, sp, t)
    int n_steps;
    float dt;
    const float* u_jump;   // [n_steps,B,N] or null
    uint64_t seed, jet_offset;
    int B, N;
    float *v_out, *logits_out, *hidden_out;  // forward outputs
    // generate: jets binned by tc_bin kernels — big_list [counts[0]] jets with a live particle at index >= 64 (one per tile),
    // small_list [counts[1]] the others (two per tile, 64 rows each); forward: null, jet s on tile s
    const int32_t *big_list, *small_list, *counts;
    const float* tvec;     // generate: [n_steps][2+2L][16] per-step time vectors from tc_time_vectors_kernel; forward: null
};

// per-group shared memory: A tile (4 KB), mask tile (4 KB), dynamic bias operand of local_0 (512 B)
constexpr int kGrpFixed = 4096 + 4096 + 512;

// per-group shared scratch (floats)
struct JetVec {
    float gv[16], gv2[16], xg[kGP], xgmid[kGP], skipg[kGP], bias_l1[16];
    float tv_bias0[16], tv_g0[16], tv_g1[kMaxL][16], tv_l1[kMaxL][16];
    int cnt[4];
    uint32_t live16[4];   // per row quarter: bit 0 / 1 = rows 0-15 / 16-31 of the quarter hold a live particle
};

template <int DC, int S, int SH, bool GENERATE>
__global__ void __launch_bounds__(kJPC * 128, 2) epic_tc_kernel(const TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const TcLayout& lay = p.lay;
    const int tid = threadIdx.x;
    // ---- carve
    uint8_t* s_bops = smem;                                   // n_bops * 512 B
    uint8_t* s_ones = s_bops + lay.n_bops * 512;              // 4 KB: A operand of the pooling GEMM (and of the all-row bias steps)
    uint8_t* s_ones_tb = s_ones + 4096;                       // 2 x 4 KB: ones in rows 0-63 only / rows 64-127 only (paired tiles)
    float* s_wf = reinterpret_cast<float*>(s_ones_tb + 8192); // fp32 tables
    uint8_t* s_grp = reinterpret_cast<uint8_t*>(s_wf + lay.n_floats);
    constexpr int kJV = (sizeof(JetVec) + 15) & ~15;
    constexpr int kGrpBytes = kGrpFixed + 2 * kJV + 16;   // a tile carries one jet, or two small ones (one JetVec each)
    __shared__ uint32_t s_tmem_slot;
    // binned generation: the tiles are [pairs of small jets | big jets]; CTAs past the last tile leave before any set-up
    int n_big = 0, n_small = 0;
    long n_slots = p.B;
    if constexpr (GENERATE) {
        n_big = __ldg(p.counts);
        n_small = __ldg(p.counts + 1);
        n_slots = (long)n_big + (n_small + 1) / 2;
        if ((long)blockIdx.x * kJPC >= n_slots) return;
    }

    // ---- one-time: weights -> smem, ones, barriers, TMEM
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.image);
        uint4* dst = reinterpret_cast<uint4*>(smem);
        const int n16 = lay.n_bops * 32;  // 512 B per operand
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = __ldg(src + i);
        const uint4* srcf = reinterpret_cast<const uint4*>(p.image + lay.n_bops * 512);
        uint4* dstf = reinterpret_cast<uint4*>(s_wf);
        for (int i = tid; i < lay.n_floats / 4; i += blockDim.x) dstf[i] = __ldg(srcf + i);
        const uint32_t one2 = 0x3F803F80u;  // bf16 1.0 twice
        for (int i = tid; i < 256; i += blockDim.x) reinterpret_cast<uint4*>(s_ones)[i] = make_uint4(one2, one2, one2, one2);
        for (int i = tid; i < 512; i += blockDim.x) {   // rows 8g..8g+7 of a K-major tile are the 256 bytes at 256 g
            const uint32_t v = ((i < 256) == ((i & 255) < 128)) ? one2 : 0u;
            reinterpret_cast<uint4*>(s_ones_tb)[i] = make_uint4(v, v, v, v);
        }
    }
    // warp-uniform indices come from a broadcast so that the compiler keeps everything derived from them (shared-memory
    // addresses, TMEM addresses, UMMA descriptors) in uniform registers: a tcgen05.mma whose operands are not provably uniform
    // is wrapped in an elect/broadcast loop of ~15 instructions
    const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int grp = warp_u >> 2, gt = tid & 127, wq = warp_u & 3, lane = tid & 31;
    // the "special" warp of a group issues its MMAs and runs its per-jet global MLP; warp w lives on SM sub-partition
    // w % 4, so rotating the role with the group index spreads that serial work over all four schedulers
    const long slot = (long)blockIdx.x * kJPC + grp;
    const bool have = slot < n_slots;
    // tile -> jet(s).  `paired` feeds MMA operands, so it is broadcast; the jet ids only feed per-thread addresses and keys.
    bool paired = false;
    int jet = (int)slot;    // the jet of THIS thread's rows (-1: none); 32-bit on purpose: it stays live through the whole loop
    if constexpr (GENERATE) {
        if (have) {
            const long n_pairs = (n_small + 1) / 2;   // paired tiles take longer per step: they go first, the single-jet tiles fill the tail
            if (slot >= n_pairs) {
                jet = __ldg(p.big_list + (slot - n_pairs));
            } else {
                paired = true;
                const long t2 = 2 * slot + ((tid >> 6) & 1);   // rows 0-63: first jet of the pair, rows 64-127: second
                jet = t2 < n_small ? __ldg(p.small_list + t2) : -1;
            }
        }
    }
    paired = __shfl_sync(0xffffffffu, (int)paired, 0) != 0;
    const int half = paired ? (wq >> 1) : 0;
    const bool has_jet = have && jet >= 0;
    // Generation: a jet's particles sit live-first (prefix mask), so the row quarters 1..3 of most jets are dead.  The tile rows
    // are rotated by `rot` quarters per jet (the network is permutation-invariant; keyed by the GLOBAL jet index, so results do
    // not depend on the batch slicing): the live quarters of the four jets of a CTA land on four different SM sub-partitions,
    // warps whose 32 particles are all dead skip every epilogue (their A rows stay zero, they only keep the barriers), and the
    // special role goes to the warp of the last quarter, which is the least likely to have row work of its own.
    // A paired tile gives each jet two row quarters: the same rotation by (global jet index & 1), the special role on the jet's
    // second quarter; the special warp of the first jet issues the tile's MMAs.
    const int rot = GENERATE ? (int)((p.jet_offset + (uint64_t)(jet < 0 ? 0 : jet)) & (paired ? 1 : 3)) : 0;
    const int swq = GENERATE ? (paired ? 2 * half + ((rot + 1) & 1) : ((rot + 3) & 3)) : (grp & 3);
    const bool is_special = has_jet && wq == swq;
    const bool is_issuer = paired ? (half == 0 && wq == swq) : (wq == swq);
    uint8_t* abuf = s_grp + grp * kGrpBytes;
    uint8_t* amask = abuf + 4096;   // A tile of the bias K-steps: columns 0,1 = mask of the row's particle
    uint8_t* bb0 = abuf + 8192;     // B tile carrying this step's local_0 bias (hi, lo) in columns 0,1
    JetVec& jv = *reinterpret_cast<JetVec*>(abuf + kGrpFixed + half * kJV);     // this thread's jet
    JetVec& jv0 = *reinterpret_cast<JetVec*>(abuf + kGrpFixed);                  // tile-level fields live in the first one
    const uint32_t mbar = smem_u32(abuf + kGrpFixed + 2 * kJV);
    if (gt == 0) mbar_init(mbar, 1);
    if (tid < 32) tmem_alloc(smem_u32(&s_tmem_slot), kJPC * kTmemPerJet);
    fence_barrier_init();
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, s_tmem_slot, 0);
    const uint32_t t_main = tmem_base + grp * kTmemPerJet + ((uint32_t)(wq * 32) << 16);
    const uint32_t t_pool = t_main + 16, t_skip = t_main + 32;
    const uint32_t d_main = tmem_base + grp * kTmemPerJet, d_pool = d_main + 16;

    if (have) {
        const int N = p.N, r = gt;                       // r: tile row (TMEM lane); n: the particle it carries
        const int n = paired ? (32 * (((wq & 1) - rot) & 1) + lane) : ((r + 128 - 32 * rot) & 127);
        const bool valid = has_jet && n < N;
        const size_t pidx = (size_t)jet * N + n;   // prologue loads only; the stores at the end recompute it
        // ---- state
        float xs[DC];
        int kk = 0, m = 0;
        if (valid) {
            m = p.mask[pidx] ? 1 : 0;
            // dead particles: the first Euler step multiplies them to 0 (bridges.py:42) and nothing reads them before
#pragma unroll
            for (int c = 0; c < DC; ++c) xs[c] = m ? p.x[pidx * DC + c] : 0.0f;
            kk = m ? p.k[pidx] : 0;
        } else {
#pragma unroll
            for (int c = 0; c < DC; ++c) xs[c] = 0.0f;
        }
        const bool live = m != 0;
        {
            uint8_t* q = amask + (r >> 3) * 256 + (r & 7) * 16;
            *reinterpret_cast<uint4*>(q) = make_uint4(live ? 0x3F803F80u : 0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(q + 128) = make_uint4(0u, 0u, 0u, 0u);
            if (gt < 32) reinterpret_cast<uint4*>(bb0)[gt] = make_uint4(0u, 0u, 0u, 0u);
        }
        bool skip = false;   // this warp has no live particle: no epilogue work at all (generation only)
        {
            const unsigned bal = __ballot_sync(0xffffffffu, m);
            if (lane == 0) {
                jv.cnt[paired ? (wq & 1) : wq] = __popc(bal);
                jv0.live16[wq] = ((bal & 0xffffu) ? 1u : 0u) | ((bal >> 16) ? 2u : 0u);   // by tile quarter
            }
            if constexpr (GENERATE) {
                skip = bal == 0u;
                if (skip) {   // its A rows are never written again: zero them once
                    float zero[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) zero[i] = 0.0f;
                    store_a_row(abuf, r, zero);
                }
            }
        }
        group_bar(1 + grp);
        const int jet_cnt = paired ? jv.cnt[0] + jv.cnt[1] : jv.cnt[0] + jv.cnt[1] + jv.cnt[2] + jv.cnt[3];
        const float inv_cnt = 1.0f / (float)jet_cnt;
        const bool jet_empty = GENERATE && jet_cnt == 0;
        // K-steps of the pooling GEMM (16 particles each) that hold a live particle; the others would add zeros
        const uint32_t pool_live = __shfl_sync(0xffffffffu, GENERATE ? (jv0.live16[0] | (jv0.live16[1] << 2) | (jv0.live16[2] << 4) | (jv0.live16[3] << 6)) : 0xffu, 0);

        const uint32_t a_addr = smem_u32(abuf);
        const uint32_t bops_addr = smem_u32(s_bops);
        const uint64_t a_desc = smem_desc(a_addr, 128, 256);
        const uint64_t ones_desc = smem_desc(smem_u32(s_ones), 128, 256);
        // pooling A operand per K-step half: a paired tile sums rows 0-63 into rows 0-63 and rows 64-127 into rows 64-127
        const uint64_t pool_a_lo = paired ? smem_desc(smem_u32(s_ones_tb), 128, 256) : ones_desc;
        const uint64_t pool_a_hi = paired ? smem_desc(smem_u32(s_ones_tb + 4096), 128, 256) : ones_desc;
        const uint64_t amask_desc = smem_desc(smem_u32(amask), 128, 256);
        const uint64_t bb0_desc = smem_desc(smem_u32(bb0), 128, 256);
        const uint64_t bops_desc0 = smem_desc(bops_addr, 128, 256);
        auto bop_desc = [&](int op) { return bops_desc0 + (uint64_t)(op * 32); };   // 512 B per operand, address field is >> 4
        const uint64_t pool_desc0 = smem_desc(a_addr, 256, 128);                      // A tile re-read MN-major
        constexpr uint32_t idesc_k = instr_desc(128, 16, false);
        constexpr uint32_t idesc_pool = instr_desc(128, 16, true);
        const int n_w = lay.n_weights();
        // D = A * (Whi + Wlo)^T: two K-steps on the same A tile
        auto gemm = [&](int op) {
            umma(d_main, a_desc, bop_desc(op), idesc_k, 0);
            umma(d_main, a_desc, bop_desc(op + n_w), idesc_k, 1);
        };
        const int T = lay.T, L = lay.L;
        const int o16 = lane & 15, hf = lane >> 4;

        const int n_steps = GENERATE ? p.n_steps : 1;
        // The step loop exists twice: once for row warps (and special warps that also carry live particles), once for a special
        // warp without live particles (SOLO) — there no per-particle state is alive, so the whole register budget is free to
        // pipeline the shared-memory loads of the per-jet global MLP, the longest serial stretch of a step.  All mutable
        // per-thread state lives inside the lambda (nothing captured by reference is written).
        auto run_steps = [&](auto solo_tag, const float (&xs_in)[DC], const int kk_in) {
        // MODE 0: a warp with live particles (all row work; possibly special as well); 1: a special warp without live particles;
        // 2: neither — it only keeps the barriers.  `skip` is a compile-time fact inside each copy.
        constexpr int MODE = decltype(solo_tag)::value;
        constexpr bool ROWS = MODE == 0;
        const bool special_here = MODE == 1 ? true : (MODE == 2 ? false : is_special);
        const bool issuer_here = MODE == 2 ? false : is_issuer;
        float xs[DC];
#pragma unroll
        for (int c = 0; c < DC; ++c) xs[c] = xs_in[c];
        int kk = kk_in;
        uint32_t phase = 0;
        // MMA completion: every warp that is going to read the accumulator polls the mbarrier itself (try_wait suspends in
        // hardware, and 60 % of the issue slots are idle anyway); warps without row work, the special warp included, do not
        // wait at all — the barrier after the epilogue is what orders the next MMA behind this one's readers.
        auto wait_mma = [&]() {
            if constexpr (ROWS) mbar_wait(mbar, phase);
            phase ^= 1;
        };
        uint32_t uq0 = 0, uq1 = 0, uq2 = 0, uq3 = 0;   // this particle's jump uniforms of the current group of four steps
        for (int step = 0; step < n_steps; ++step) {
            // ---- (a) time vectors (warp 0) and the first A row [x_hi, x_lo, onehot(k)] * m
            if constexpr (GENERATE) {
                // the time is shared by all jets at generation: the vectors were computed once per step by the prologue kernel
                if (special_here) {
                    const float* tv = p.tvec + (size_t)step * (2 + 2 * L) * 16;
                    const int vi = lane >> 4;   // two vectors per pass
                    for (int v0 = 0; v0 < 2 + 2 * L; v0 += 2) {
                        const float val = __ldg(tv + (v0 + vi) * 16 + o16);
                        const int v = v0 + vi;
                        if (v == 0) {
                            const float hi = __bfloat162float(__float2bfloat16_rn(val));
                            *reinterpret_cast<uint32_t*>(bb0 + (o16 >> 3) * 256 + (o16 & 7) * 16) = pack_bf16(hi, val - hi);
                        } else if (v == 1) jv.tv_g0[o16] = val;
                        else if ((v & 1) == 0) jv.tv_g1[(v - 2) >> 1][o16] = val;
                        else jv.tv_l1[(v - 2) >> 1][o16] = val;
                    }
                }
            } else if (special_here) {
                const float* te = p.temb + (size_t)jet * p.temb_stride;
                const int t0 = hf * (T / 2), t1 = t0 + T / 2;
                float a0 = hf ? 0.0f : s_wf[lay.c0 + o16], a1 = hf ? 0.0f : s_wf[lay.g0b + o16];
                for (int t = t0; t < t1; ++t) {
                    const float tv = __ldg(te + t);
                    a0 = fmaf(s_wf[lay.w0t + t * 16 + o16], tv, a0);
                    a1 = fmaf(s_wf[lay.g0t + t * 16 + o16], tv, a1);
                }
                a0 += __shfl_xor_sync(0xffffffffu, a0, 16);
                a1 += __shfl_xor_sync(0xffffffffu, a1, 16);
                if (hf == 0) {
                    const float hi = __bfloat162float(__float2bfloat16_rn(a0));
                    *reinterpret_cast<uint32_t*>(bb0 + (o16 >> 3) * 256 + (o16 & 7) * 16) = pack_bf16(hi, a0 - hi);
                    jv.tv_g0[o16] = a1;
                }
                for (int l = 0; l < L; ++l) {
                    const float* Wl = s_wf + lay.layer0 + l * lay.layer_stride;
                    float b0 = hf ? 0.0f : Wl[lay.l_g1b + o16], b1 = hf ? 0.0f : Wl[lay.l_l1b + o16];
                    for (int t = t0; t < t1; ++t) {
                        const float tv = __ldg(te + t);
                        b0 = fmaf(Wl[lay.l_g1t + t * 16 + o16], tv, b0);
                        b1 = fmaf(Wl[lay.l_l1t + t * 16 + o16], tv, b1);
                    }
                    b0 += __shfl_xor_sync(0xffffffffu, b0, 16);
                    b1 += __shfl_xor_sync(0xffffffffu, b1, 16);
                    if (hf == 0) { jv.tv_g1[l][o16] = b0; jv.tv_l1[l][o16] = b1; }
                }
            }
            if constexpr (ROWS) {
                float row[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) row[i] = 0.0f;
#pragma unroll
                for (int c = 0; c < DC; ++c) {
                    const float hi = __bfloat162float(__float2bfloat16_rn(xs[c]));
                    row[c] = hi;
                    row[DC + c] = xs[c] - hi;
                }
#pragma unroll
                for (int s = 0; s < S; ++s) row[2 * DC + s] = (kk == s) ? 1.0f : 0.0f;
                store_a_row_masked(abuf, r, row, live);
            }
            fence_proxy_async();
            group_bar(1 + grp);
            // ---- (b) local_0
            if (issuer_here && elect_one()) {
                tc_fence_after();
                gemm(lay.bop_local0());
                umma(d_main, amask_desc, bb0_desc, idesc_k, 1);  // + bias on live rows; dead rows stay exactly 0
                umma_commit(mbar);
            }
            wait_mma();
            tc_fence_after();
            float acc[16], xl[16];
            if constexpr (ROWS) {
                tmem_ld16(t_main, acc);
                lrelu16(xl, acc);
                if (lay.skip) tmem_st16(t_skip, xl);   // x_local_skip (epic.py:148) parked in TMEM, not in registers
                store_a_row(abuf, r, xl);
            }
            tc_fence_before();
            fence_proxy_async();
            group_bar(1 + grp);

            for (int l = 0; l < L; ++l) {
                const float* Wl = s_wf + lay.layer0 + l * lay.layer_stride;
                // ---- (d) pooling GEMM (ones x XL, K = 128 particles) + fc_local1 on the same tile
                if (issuer_here && elect_one()) {
                    tc_fence_after();
                    umma_pool8(d_pool, pool_a_lo, pool_a_hi, pool_desc0, idesc_pool, pool_live);  // K-step j = rows 16j..16j+15, MN-major
                    gemm(lay.bop_l1(l));
                    umma_commit(mbar);
                }
                phase ^= 1;
                // ---- (e) global path on warp 0 of the group (fp32, CUDA cores); the other warps park at the barrier below
                if (special_here) {
                    mbar_wait(mbar, phase ^ 1);
                    tc_fence_after();
                    float sv[16];
                    tmem_ld16(t_pool, sv);
                    if (l == 0) {  // EPiC_Projection globals (epic.py:187-190)
                        float g = hf ? 0.0f : jv.tv_g0[o16];
                        const float sc = hf ? 1.0f : inv_cnt;
                        g = dotr16(g, s_wf + lay.g0ms + o16 * kS32 + hf * 16, sv, sc);
                        g += __shfl_xor_sync(0xffffffffu, g, 16);
                        if (hf == 0) jv.gv[o16] = lrelu_fast(g);
                        __syncwarp();
                        g = hf ? 0.0f : s_wf[lay.g1b + o16];
                        g = dotv<8>(g, s_wf + lay.g1 + o16 * kS16 + hf * 8, jv.gv + hf * 8);
                        g += __shfl_xor_sync(0xffffffffu, g, 16);
                        if (hf == 0) jv.gv2[o16] = lrelu_fast(g);
                        __syncwarp();
                        g = s_wf[lay.g2b + lane];
                        g = dotv<16>(g, s_wf + lay.g2 + lane * kS16, jv.gv2);
                        g = lrelu_fast(g);
                        jv.xg[lane] = g;
                        jv.skipg[lane] = lay.skip ? g : 0.0f;
                        __syncwarp();
                    }
                    // EPiC_layer globals (epic.py:228-232)
                    float g = hf ? 0.0f : jv.tv_g1[l][o16];
                    g = dotr16(g, Wl + lay.l_g1ms + o16 * kS32 + hf * 16, sv, hf ? 1.0f : inv_cnt);
                    g = dotv<kGP / 2>(g, Wl + lay.l_g1g + o16 * kS32 + hf * (kGP / 2), jv.xg + hf * (kGP / 2));
                    g += __shfl_xor_sync(0xffffffffu, g, 16);
                    __syncwarp();
                    if (hf == 0) jv.gv[o16] = lrelu_fast(g);
                    __syncwarp();
                    g = Wl[lay.l_g2b + lane];
                    g = dotv<16>(g, Wl + lay.l_g2 + lane * kS16, jv.gv);
                    const float xmid = lrelu_fast(g + jv.xg[lane]);
                    __syncwarp();
                    jv.xgmid[lane] = xmid;
                    jv.xg[lane] = xmid + jv.skipg[lane];
                    __syncwarp();
                    // per-jet bias of fc_local1: time part + Wl1[:, H:H+G] xg   (epic.py:233-238)
                    g = hf ? 0.0f : jv.tv_l1[l][o16];
                    g = dotv<kGP / 2>(g, Wl + lay.l_l1g + o16 * kS32 + hf * (kGP / 2), jv.xgmid + hf * (kGP / 2));
                    g += __shfl_xor_sync(0xffffffffu, g, 16);
                    if (hf == 0) jv.bias_l1[o16] = g;
                    tc_fence_before();
                }
                group_bar(1 + grp);
                // ---- (f) fc_local1 epilogue -> A operand of fc_local2
                tc_fence_after();
                if constexpr (ROWS) {
                    tmem_ld16(t_main, acc);
                    float l1[16], bl[16];
                    lds16(jv.bias_l1, bl);
                    lrelu16_sum(l1, acc, bl);
                    store_a_row(abuf, r, l1);
                }
                tc_fence_before();
                fence_proxy_async();
                group_bar(1 + grp);
                // ---- (g) fc_local2
                if (issuer_here && elect_one()) {
                    tc_fence_after();
                    gemm(lay.bop_l2(l));
                    umma(d_main, amask_desc, bop_desc(lay.bop_bias_l2(l)), idesc_k, 1);
                    umma_commit(mbar);
                }
                wait_mma();
                tc_fence_after();
                if constexpr (ROWS) {
                    tmem_ld16(t_main, acc);
                    lrelu16_sum(xl, acc, xl);  // dead rows: unused garbage, zeroed at pack
                    if (lay.skip) {
                        tmem_ld16(t_skip, acc);
#pragma unroll
                        for (int i = 0; i < 16; i += 2) fadd2(xl[i], xl[i + 1], xl[i], xl[i + 1], acc[i], acc[i + 1]);
                    }
                    store_a_row_masked(abuf, r, xl, live);
                }
                tc_fence_before();
                fence_proxy_async();
                group_bar(1 + grp);
            }
            // ---- (i) output layer (epic.py:158-162)
            if (issuer_here && elect_one()) {
                tc_fence_after();
                // with a discrete head the operand is [W_out(v rows) ; F1 W_out(z rows)]: the output layer and the first
                // head Linear have no nonlinearity between them, so columns DC.. are already F1 z + f1 (mbm.py:105-111)
                gemm(lay.bop_out());
                umma(d_main, amask_desc, bop_desc(lay.bop_bias_out()), idesc_k, 1);  // live rows: b_out | F1 b_out_z
                if constexpr (SH > 0) umma(d_main, ones_desc, bop_desc(lay.bop_bias_h0()), idesc_k, 1);  // all rows: f1 (fc(0) on dead rows)
                umma_commit(mbar);
            }
            wait_mma();
            tc_fence_after();
            float h[16];
            if constexpr (ROWS) tmem_ld16(t_main, h);   // h[0..DC) = velocity (0 on dead rows); h[DC..) = head pre-activation or raw logits
            float lg[S];
            if constexpr (SH > 0) {
                if constexpr (ROWS) {
                    float z1[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) z1[i] = i < SH ? selu_fast(h[DC + (i < SH ? i : 0)]) : 0.0f;
                    store_a_row(abuf, r, z1);
                }
                tc_fence_before();
                fence_proxy_async();
                group_bar(1 + grp);
                if (issuer_here && elect_one()) {
                    tc_fence_after();
                    gemm(lay.bop_h2());
                    umma(d_main, ones_desc, bop_desc(lay.bop_bias_h2()), idesc_k, 1);
                    umma_commit(mbar);
                }
                wait_mma();
                tc_fence_after();
                if constexpr (!ROWS) {
                } else if constexpr (S <= 8) {
                    float l8[8];
                    tmem_ld8(t_main, l8);
#pragma unroll
                    for (int s = 0; s < S; ++s) lg[s] = l8[s];
                } else {
                    tmem_ld16(t_main, acc);
#pragma unroll
                    for (int s = 0; s < S; ++s) lg[s] = acc[s];
                }
            } else {
#pragma unroll
                for (int s = 0; s < S; ++s) lg[s] = h[DC + s];
            }
            tc_fence_before();  // orders this step's last tcgen05.ld before the next step's first MMA (via the group barrier)

            if constexpr (GENERATE && ROWS) {
                // ---- (k) hybrid update in registers (bridges.py:38-45,179-201)
                const StepScalars sc{p.dt, __ldg(p.step_tab + step * 4 + 0), __ldg(p.step_tab + step * 4 + 1), 0.0f};
#pragma unroll
                for (int c = 0; c < DC; ++c) xs[c] = fmaf(p.dt, h[c], xs[c]);  // h = 0 on dead rows, x there stays 0
                // One Philox block carries the uniforms of four consecutive particles at one step.  Instead of every lane
                // recomputing the block of its quad each step, lane j of a quad generates the block of step (s & ~3) + j once per
                // four steps and a 4 x 4 transpose inside the quad (four shuffles) hands every lane its own word of each step:
                // the same (seed, jet, step, particle) -> uniform map as philox_uniform(), a quarter of the arithmetic.
                if (!p.u_jump && (step & 3) == 0) {
                    const uint4 blk = philox_block(p.seed, p.jet_offset + (uint64_t)jet, 0, step + (n & 3), n >> 2);
                    uint32_t a0 = blk.x, a1 = blk.y, a2 = blk.z, a3 = blk.w;
                    {   // exchange 2 x 2 blocks with lane ^ 2
                        const bool hi = (lane & 2) != 0;
                        const uint32_t r0 = __shfl_xor_sync(0xffffffffu, hi ? a0 : a2, 2), r1 = __shfl_xor_sync(0xffffffffu, hi ? a1 : a3, 2);
                        if (hi) { a0 = r0; a1 = r1; } else { a2 = r0; a3 = r1; }
                    }
                    {   // then single elements with lane ^ 1
                        const bool hi = (lane & 1) != 0;
                        const uint32_t r0 = __shfl_xor_sync(0xffffffffu, hi ? a0 : a1, 1), r1 = __shfl_xor_sync(0xffffffffu, hi ? a2 : a3, 1);
                        if (hi) { a0 = r0; a2 = r1; } else { a1 = r0; a3 = r1; }
                    }
                    uq0 = a0; uq1 = a1; uq2 = a2; uq3 = a3;   // word (r & 3) of the blocks of steps s, s+1, s+2, s+3
                }
                if (valid) {
                    const int ph = step & 3;
                    const float u = p.u_jump ? __ldg(p.u_jump + ((size_t)step * p.B + jet) * N + n)
                                             : u01(ph == 0 ? uq0 : ph == 1 ? uq1 : ph == 2 ? uq2 : uq3);
                    kk = telegraph_jump_fast<S>(lg, kk, u, sc) * m;
                }
            }
            if constexpr (!GENERATE) {
                if (valid) {
                    const size_t pout = (size_t)jet * p.N + n;
#pragma unroll
                    for (int c = 0; c < DC; ++c) p.v_out[pout * DC + c] = h[c];
#pragma unroll
                    for (int s = 0; s < S; ++s) p.logits_out[pout * S + s] = lg[s];
                    if (p.hidden_out) {
#pragma unroll
                        for (int i = 0; i < 16; i += 4)
                            *reinterpret_cast<float4*>(p.hidden_out + pout * 16 + i) =
                                live ? make_float4(xl[i], xl[i + 1], xl[i + 2], xl[i + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
            }
        }
        if constexpr (GENERATE) {
            if (valid) {
                const size_t pout = (size_t)jet * p.N + n;
                // an empty jet ends as in the reference: mean pool 0/0 (epic.py:141) -> NaN velocity -> (x + dt NaN) * 0 = NaN
                // for every particle (bridges.py:42); tokens are integers times the mask = 0
                const float dead_x = jet_empty ? __int_as_float(0x7fc00000) : 0.0f;
#pragma unroll
                for (int c = 0; c < DC; ++c) p.x[pout * DC + c] = jet_empty ? dead_x : xs[c];
                p.k[pout] = (uint8_t)kk;
                if (paired && n + 64 < p.N) {   // a small jet's particles 64.. are dead and have no row in a paired tile: final state 0
#pragma unroll
                    for (int c = 0; c < DC; ++c) p.x[(pout + 64) * DC + c] = dead_x;
                    p.k[pout + 64] = 0;
                }
            }
        }
        };
        if (!skip) run_steps(std::integral_constant<int, 0>{}, xs, kk);
        else if (is_special) run_steps(std::integral_constant<int, 1>{}, xs, kk);
        else run_steps(std::integral_constant<int, 2>{}, xs, kk);
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 32) tmem_dealloc(tmem_base, kJPC * kTmemPerJet);
}

size_t tc_smem_bytes(const TcLayout& lay) {
    const size_t grp = kGrpFixed + 2 * ((sizeof(JetVec) + 15) & ~15) + 16;
    return (size_t)lay.n_bops * 512 + 4096 + 8192 + (size_t)lay.n_floats * 4 + kJPC * grp + 1024;
}

template <int DC, int S, int SH, bool GEN>
int launch(const TcParams& p, cudaStream_t stream) {
    const size_t bytes = tc_smem_bytes(p.lay);
    auto kern = epic_tc_kernel<DC, S, SH, GEN>;
    if (int rc = cuda_ok(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), "tc smem attribute")) return rc;
    const int grid = (p.B + kJPC - 1) / kJPC;
    kern<<<grid, kJPC * 128, bytes, stream>>>(p);
    return cuda_ok(cudaGetLastError(), "epic_tc launch");
}

template <bool GEN>
int dispatch(const MmbEpicDims& d, const TcParams& p, cudaStream_t stream) {
    const int sh = d.disc_head_hidden;
    if (d.dim_continuous == 3 && d.vocab_size == 8 && sh == 8) return launch<3, 8, 8, GEN>(p, stream);
    if (d.dim_continuous == 3 && d.vocab_size == 8 && sh == 0) return launch<3, 8, 0, GEN>(p, stream);
    if (d.dim_continuous == 3 && d.vocab_size == 4 && sh == 4) return launch<3, 4, 4, GEN>(p, stream);
    if (d.dim_continuous == 3 && d.vocab_size == 4 && sh == 0) return launch<3, 4, 0, GEN>(p, stream);
    return fail(MMB_EUNSUPPORTED, "tcgen05 path instantiated for (Dc,S,head) in {(3,8,8),(3,8,0),(3,4,4),(3,4,0)}");
}

}  // namespace

// the fused discrete head handles Sh == S (MultiModalEPiC.fc_layer); any other width (AbsorbingGenerator's 56) runs
// the tensor-core trunk headless and a small per-particle MLP kernel on its logit slice
static bool head_fused(const MmbEpicDims& d) { return d.disc_head_hidden == 0 || d.disc_head_hidden == d.vocab_size; }
static MmbEpicDims tc_dims(const MmbEpicDims& d) {
    MmbEpicDims t = d;
    if (!head_fused(d)) t.disc_head_hidden = 0;
    return t;
}

// logits <- W2 selu(W1 z + b1) + b2 in place, z = logits (the raw output-layer slice)   (absorbing_flows.py:41-54,133-138)
template <int S>
__global__ void __launch_bounds__(256) discrete_head_mlp_kernel(const float* __restrict__ W, MmbEpicLayout Lo, int Sh,
                                                                float* __restrict__ logits, size_t P) {
    // W1 [Sh][S] | b1 [Sh, padded to a multiple of 4] | W2^T [Sh][S] | b2 [S]: every weight row starts on 16 bytes
    extern __shared__ __align__(16) float sw[];
    const int ShP = (Sh + 3) & ~3, oB1 = Sh * S, oW2 = oB1 + ShP, oB2 = oW2 + Sh * S;
    for (int i = threadIdx.x; i < Sh * S; i += blockDim.x) {
        sw[i] = __ldg(W + Lo.head0_w + i);
        const int s = i / Sh, j = i % Sh;                       // head2_w is [S][Sh]
        sw[oW2 + j * S + s] = __ldg(W + Lo.head2_w + i);
    }
    for (int i = threadIdx.x; i < Sh; i += blockDim.x) sw[oB1 + i] = __ldg(W + Lo.head0_b + i);
    for (int i = threadIdx.x; i < S; i += blockDim.x) sw[oB2 + i] = __ldg(W + Lo.head2_b + i);
    __syncthreads();
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    float z[S], out[S];
    // a particle's S logits are 16 / 32 contiguous bytes: 128-bit loads and stores when the caller's buffer allows; the weight
    // rows in shared memory are read as float4 (every lane reads the same address: one broadcast per 4 weights)
    const bool vec = (reinterpret_cast<uintptr_t>(logits) & 15) == 0;
    float4* io = reinterpret_cast<float4*>(logits + p * S);
    if (vec) {
#pragma unroll
        for (int q = 0; q < S / 4; ++q) {
            const float4 t = io[q];
            z[4 * q] = t.x; z[4 * q + 1] = t.y; z[4 * q + 2] = t.z; z[4 * q + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int s = 0; s < S; ++s) z[s] = logits[p * S + s];
    }
#pragma unroll
    for (int s = 0; s < S; ++s) out[s] = sw[oB2 + s];
    const float4* w1 = reinterpret_cast<const float4*>(sw);
    const float4* w2 = reinterpret_cast<const float4*>(sw + oW2);
#pragma unroll 4
    for (int j = 0; j < Sh; ++j) {
        float a = sw[oB1 + j];
#pragma unroll
        for (int q = 0; q < S / 4; ++q) {
            const float4 w = w1[j * (S / 4) + q];
            a = fmaf(w.x, z[4 * q], a); a = fmaf(w.y, z[4 * q + 1], a); a = fmaf(w.z, z[4 * q + 2], a); a = fmaf(w.w, z[4 * q + 3], a);
        }
        a = a > 0.0f ? 1.0507009873554805f * a : 1.7580993408473766f * (__expf(a) - 1.0f);
#pragma unroll
        for (int q = 0; q < S / 4; ++q) {
            const float4 w = w2[j * (S / 4) + q];
            out[4 * q] = fmaf(w.x, a, out[4 * q]); out[4 * q + 1] = fmaf(w.y, a, out[4 * q + 1]);
            out[4 * q + 2] = fmaf(w.z, a, out[4 * q + 2]); out[4 * q + 3] = fmaf(w.w, a, out[4 * q + 3]);
        }
    }
    if (vec) {
#pragma unroll
        for (int q = 0; q < S / 4; ++q) io[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
    } else {
#pragma unroll
        for (int s = 0; s < S; ++s) logits[p * S + s] = out[s];
    }
}

static int launch_discrete_head_mlp(const EpicModel* m, float* logits, size_t P, cudaStream_t stream) {
    const int S = m->dims.vocab_size, Sh = m->dims.disc_head_hidden;
    const size_t bytes = (size_t)(2 * Sh * S + ((Sh + 3) & ~3) + S) * sizeof(float);
    const unsigned grid = (unsigned)((P + 255) / 256);
    if (S == 8) discrete_head_mlp_kernel<8><<<grid, 256, bytes, stream>>>(m->w, m->layout, Sh, logits, P);
    else discrete_head_mlp_kernel<4><<<grid, 256, bytes, stream>>>(m->w, m->layout, Sh, logits, P);
    return cuda_ok(cudaGetLastError(), "discrete_head_mlp launch");
}

// Per-step time vectors of the generation loop (same for every jet): v0 = local_0 bias c0 + W0t temb, v1 = G0 bias + G0t temb,
// then per layer (fc_global1 bias + time part, fc_local1 bias + time part).  One block per step, one thread per output.
__global__ void tc_time_vectors_kernel(const uint8_t* __restrict__ image, TcLayout lay, const float* __restrict__ temb, float* __restrict__ tvec) {
    const float* wf = reinterpret_cast<const float*>(image + lay.n_bops * 512);
    const int step = blockIdx.x, v = threadIdx.x >> 4, o = threadIdx.x & 15;
    if (v >= 2 + 2 * lay.L) return;
    const float* te = temb + (size_t)step * lay.T;
    int base, mat;
    if (v == 0) { base = lay.c0; mat = lay.w0t; }
    else if (v == 1) { base = lay.g0b; mat = lay.g0t; }
    else {
        const int lo = lay.layer0 + ((v - 2) >> 1) * lay.layer_stride;
        base = lo + ((v & 1) ? lay.l_l1b : lay.l_g1b);
        mat = lo + ((v & 1) ? lay.l_l1t : lay.l_g1t);
    }
    // same split-in-halves summation order as the in-kernel path (two partial sums over t, then added)
    float a0 = wf[base + o], a1 = 0.0f;
    for (int t = 0; t < lay.T / 2; ++t) a0 = fmaf(wf[mat + t * 16 + o], te[t], a0);
    for (int t = lay.T / 2; t < lay.T; ++t) a1 = fmaf(wf[mat + t * 16 + o], te[t], a1);
    tvec[((size_t)step * (2 + 2 * lay.L) + v) * 16 + o] = a0 + a1;
}

// ---- binning of the jets of a generation call: "small" = no live particle at index >= 64 (two of them share a tile) ---------
// Order-preserving (deterministic) compaction in three small kernels: per-block counts, a one-warp scan, the fill.
constexpr int kBinThreads = 256;
constexpr int kPairRows = kRows / 2;   // rows of a small jet in a paired tile
__global__ void __launch_bounds__(kBinThreads) tc_bin_count_kernel(const uint8_t* __restrict__ mask, int B, int N, int vec_ok, uint8_t* __restrict__ flag,
                                                                   int32_t* __restrict__ block_small) {
    const int jet = blockIdx.x * kBinThreads + threadIdx.x;
    int small = 0;
    if (jet < B) {
        small = 1;
        const uint8_t* row = mask + (size_t)jet * N;
        if (vec_ok) {
            for (int n = kPairRows; n < N; n += 16) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(row + n));
                if (q.x | q.y | q.z | q.w) small = 0;
            }
        } else {
            for (int n = kPairRows; n < N; ++n) if (row[n]) small = 0;
        }
        flag[jet] = (uint8_t)small;
    }
    const int c = __syncthreads_count(small);
    if (threadIdx.x == 0) block_small[blockIdx.x] = c;
}
__global__ void tc_bin_scan_kernel(const int32_t* __restrict__ block_small, int nblocks, int B, int32_t* __restrict__ block_off,
                                   int32_t* __restrict__ counts) {
    const int lane = threadIdx.x;   // one warp
    int carry = 0;
    for (int base = 0; base < nblocks; base += 32) {
        const int i = base + lane;
        const int v = i < nblocks ? block_small[i] : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (i < nblocks) block_off[i] = carry + inc - v;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) { counts[0] = B - carry; counts[1] = carry; }
}
__global__ void __launch_bounds__(kBinThreads) tc_bin_fill_kernel(const uint8_t* __restrict__ flag, const int32_t* __restrict__ block_off, int B,
                                                                  int32_t* __restrict__ small_list, int32_t* __restrict__ big_list) {
    __shared__ int warp_small[kBinThreads / 32];
    const int jet = blockIdx.x * kBinThreads + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool in = jet < B;
    const bool small = in && flag[jet] != 0;
    const unsigned bs = __ballot_sync(0xffffffffu, small);
    if (lane == 0) warp_small[w] = __popc(bs);
    __syncthreads();
    int small_before = 0;
    for (int i = 0; i < w; ++i) small_before += warp_small[i];
    small_before += __popc(bs & ((1u << lane) - 1u));
    if (!in) return;
    const int off = block_off[blockIdx.x];
    if (small) small_list[off + small_before] = jet;
    else big_list[(blockIdx.x * kBinThreads - off) + (threadIdx.x - small_before)] = jet;
}
struct BinLayout {   // in 4-byte units after the time vectors
    size_t counts, block_small, block_off, small_list, big_list, flag, total;
    int nblocks;
    explicit BinLayout(int B) {
        nblocks = (B + kBinThreads - 1) / kBinThreads;
        size_t at = 0;
        auto take = [&](size_t n) { const size_t o = at; at += (n + 3) & ~(size_t)3; return o; };
        counts = take(4); block_small = take(nblocks); block_off = take(nblocks); small_list = take(B); big_list = take(B);
        flag = take(((size_t)B + 3) / 4);
        total = at;
    }
};

size_t tc_generate_scratch_floats(const MmbEpicDims* d, int n_steps, int B) {
    return (((size_t)n_steps * (2 + 2 * d->num_blocks) * 16 + 3) & ~(size_t)3) + BinLayout(B > 0 ? B : 0).total;
}

bool tc_supported(const MmbEpicDims* d, int N) {
    return d->dim_hidden_local == kH && d->dim_hidden_glob <= kGP && d->dim_time_emb <= kMaxT && d->dim_time_emb % 2 == 0 &&
           d->num_blocks >= 1 && d->num_blocks <= kMaxL && d->dim_continuous == 3 &&
           (d->vocab_size == 8 || d->vocab_size == 4) && d->disc_head_hidden <= 256 && N <= kRows && N >= 1 &&
           d->dim_context == 0;   // models with context features run on the fp32 kernel or the warp-MMA engine
}

// Build the device image from the packed fp32 blob (host): bf16 UMMA operands + fp32 side tables.
int tc_build_image(EpicModel* m, const float* W) {
    const MmbEpicDims d = tc_dims(m->dims);
    const MmbEpicLayout& Lo = m->layout;
    const TcLayout lay = make_layout(d);
    const int Dc = d.dim_continuous, S = d.vocab_size, T = d.dim_time_emb, C = d.dim_cont_emb, D = d.dim_disc_emb,
              H = kH, G = d.dim_hidden_glob, L = d.num_blocks, Sh = d.disc_head_hidden;
    const int K0 = T + C + D;
    std::vector<__nv_bfloat16> bops((size_t)lay.n_bops * 256, __float2bfloat16(0.0f));
    std::vector<float> wf((size_t)lay.n_floats, 0.0f);
    auto setb = [&](int op, int row, int k, double v) {
        const __nv_bfloat16 hi = __float2bfloat16((float)v);
        bops[(size_t)op * 256 + bop_index(row, k)] = hi;
        bops[(size_t)(op + lay.n_weights()) * 256 + bop_index(row, k)] = __float2bfloat16((float)(v - (double)__bfloat162float(hi)));
    };

    // local_0 folded: columns [x_hi | x_lo | onehot]
    for (int o = 0; o < H; ++o) {
        const float* w0 = W + Lo.local0_w + (size_t)o * K0;
        for (int j = 0; j < Dc; ++j) {
            double acc = 0;
            for (int c = 0; c < C; ++c) acc += (double)w0[T + c] * W[Lo.emb_cont_w + (size_t)c * Dc + j];
            setb(lay.bop_local0(), o, j, acc);
            setb(lay.bop_local0(), o, Dc + j, acc);
        }
        for (int s = 0; s < S; ++s) {
            double acc = 0;
            for (int dd = 0; dd < D; ++dd) acc += (double)w0[T + C + dd] * W[Lo.emb_disc + (size_t)s * D + dd];
            setb(lay.bop_local0(), o, 2 * Dc + s, acc);
        }
        double c0 = W[Lo.local0_b + o];
        for (int c = 0; c < C; ++c) c0 += (double)w0[T + c] * W[Lo.emb_cont_b + c];
        wf[lay.b0 + o] = W[Lo.local0_b + o];
        wf[lay.c0 + o] = (float)c0;
        for (int t = 0; t < T; ++t) wf[lay.w0t + t * 16 + o] = w0[t];
        // projection globals
        const float* g0 = W + Lo.global0_w + (size_t)o * (2 * H + T);
        for (int k = 0; k < H; ++k) { wf[lay.g0ms + o * kS32 + k] = g0[k]; wf[lay.g0ms + o * kS32 + 16 + k] = g0[H + k]; }
        for (int t = 0; t < T; ++t) wf[lay.g0t + t * 16 + o] = g0[2 * H + t];
        wf[lay.g0b + o] = W[Lo.global0_b + o];
        for (int k = 0; k < H; ++k) wf[lay.g1 + o * kS16 + k] = W[Lo.global1_w + (size_t)o * H + k];
        wf[lay.g1b + o] = W[Lo.global1_b + o];
    }
    for (int g = 0; g < G; ++g) {
        for (int k = 0; k < H; ++k) wf[lay.g2 + g * kS16 + k] = W[Lo.global2_w + (size_t)g * H + k];
        wf[lay.g2b + g] = W[Lo.global2_b + g];
    }
    for (int l = 0; l < L; ++l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        float* F = wf.data() + lay.layer0 + (size_t)l * lay.layer_stride;
        const int Kg = 2 * H + G + T, Kl = H + G + T;
        for (int o = 0; o < H; ++o) {
            const float* g1 = Wl + Lo.l_g1_w + (size_t)o * Kg;
            for (int k = 0; k < H; ++k) { F[lay.l_g1ms + o * kS32 + k] = g1[k]; F[lay.l_g1ms + o * kS32 + 16 + k] = g1[H + k]; }
            for (int g = 0; g < G; ++g) F[lay.l_g1g + o * kS32 + g] = g1[2 * H + g];
            for (int t = 0; t < T; ++t) F[lay.l_g1t + t * 16 + o] = g1[2 * H + G + t];
            F[lay.l_g1b + o] = Wl[Lo.l_g1_b + o];
            const float* l1 = Wl + Lo.l_l1_w + (size_t)o * Kl;
            for (int k = 0; k < H; ++k) setb(lay.bop_l1(l), o, k, l1[k]);
            for (int g = 0; g < G; ++g) F[lay.l_l1g + o * kS32 + g] = l1[H + g];
            for (int t = 0; t < T; ++t) F[lay.l_l1t + t * 16 + o] = l1[H + G + t];
            F[lay.l_l1b + o] = Wl[Lo.l_l1_b + o];
            for (int k = 0; k < H; ++k) setb(lay.bop_l2(l), o, k, Wl[Lo.l_l2_w + (size_t)o * H + k]);
            F[lay.l_l2b + o] = Wl[Lo.l_l2_b + o];
        }
        for (int g = 0; g < G; ++g) {
            for (int k = 0; k < H; ++k) F[lay.l_g2 + g * kS16 + k] = Wl[Lo.l_g2_w + (size_t)g * H + k];
            F[lay.l_g2b + g] = Wl[Lo.l_g2_b + g];
        }
    }
    if (!Sh) {
        for (int o = 0; o < Dc + S; ++o)
            for (int k = 0; k < H; ++k) setb(lay.bop_out(), o, k, W[Lo.out_w + (size_t)o * H + k]);
    } else {  // rows [0,Dc): output layer (velocity); rows [Dc,Dc+Sh): head Linear 0 folded through the output layer
        for (int o = 0; o < Dc; ++o)
            for (int k = 0; k < H; ++k) setb(lay.bop_out(), o, k, W[Lo.out_w + (size_t)o * H + k]);
        for (int j = 0; j < Sh; ++j)
            for (int k = 0; k < H; ++k) {
                double acc = 0;
                for (int s = 0; s < S; ++s) acc += (double)W[Lo.head0_w + (size_t)j * S + s] * W[Lo.out_w + (size_t)(Dc + s) * H + k];
                setb(lay.bop_out(), Dc + j, k, acc);
            }
        for (int o = 0; o < S; ++o) {
            for (int k = 0; k < Sh; ++k) setb(lay.bop_h2(), o, k, W[Lo.head2_w + (size_t)o * Sh + k]);
            wf[lay.bh2 + o] = W[Lo.head2_b + o];
        }
    }
    auto set_bias = [&](int op, int o, float b) {
        const __nv_bfloat16 hi = __float2bfloat16(b);
        bops[(size_t)op * 256 + bop_index(o, 0)] = hi;
        bops[(size_t)op * 256 + bop_index(o, 1)] = __float2bfloat16(b - __bfloat162float(hi));
    };
    for (int l = 0; l < L; ++l)
        for (int o = 0; o < H; ++o) set_bias(lay.bop_bias_l2(l), o, W[Lo.layer0 + (size_t)l * Lo.layer_stride + Lo.l_l2_b + o]);
    if (!Sh) {
        for (int o = 0; o < Dc + S; ++o) set_bias(lay.bop_bias_out(), o, W[Lo.out_b + o]);
    } else {
        for (int o = 0; o < Dc; ++o) set_bias(lay.bop_bias_out(), o, W[Lo.out_b + o]);
        for (int j = 0; j < Sh; ++j) {
            double acc = 0;
            for (int s = 0; s < S; ++s) acc += (double)W[Lo.head0_w + (size_t)j * S + s] * W[Lo.out_b + Dc + s];
            set_bias(lay.bop_bias_out(), Dc + j, (float)acc);
            set_bias(lay.bop_bias_h0(), Dc + j, W[Lo.head0_b + j]);
        }
        for (int o = 0; o < S; ++o) set_bias(lay.bop_bias_h2(), o, W[Lo.head2_b + o]);
    }
    const size_t nb = bops.size() * sizeof(__nv_bfloat16), nf = wf.size() * sizeof(float);
    m->tc_image_bytes = nb + nf;
    if (int rc = cuda_ok(cudaMalloc(&m->tc_image, m->tc_image_bytes), "cudaMalloc tc image")) return rc;
    if (int rc = cuda_ok(cudaMemcpy(m->tc_image, bops.data(), nb, cudaMemcpyHostToDevice), "tc image upload")) return rc;
    return cuda_ok(cudaMemcpy(static_cast<uint8_t*>(m->tc_image) + nb, wf.data(), nf, cudaMemcpyHostToDevice), "tc image upload");
}

int launch_epic_forward_tc(const EpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask,
                           const float* temb, int temb_stride, int B, int N,
                           float* v_out, float* logits_out, float* hidden_out, cudaStream_t stream) {
    if (B == 0) return MMB_OK;
    TcParams p{};
    p.image = static_cast<const uint8_t*>(m->tc_image);
    p.lay = make_layout(tc_dims(m->dims));
    p.x = const_cast<float*>(x); p.k = const_cast<uint8_t*>(k); p.mask = mask;
    p.temb = temb; p.temb_stride = temb_stride; p.n_steps = 1;
    p.B = B; p.N = N; p.v_out = v_out; p.logits_out = logits_out; p.hidden_out = hidden_out;
    if (int rc = dispatch<false>(tc_dims(m->dims), p, stream)) return rc;
    return head_fused(m->dims) ? MMB_OK : launch_discrete_head_mlp(m, logits_out, (size_t)B * N, stream);
}

int launch_generate_tc(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* dev_table, float* scratch,
                       int n_steps, float dt, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                       int B, int N, cudaStream_t stream) {
    if (B == 0 || n_steps == 0) return MMB_OK;
    if (!head_fused(m->dims)) return fail(MMB_EUNSUPPORTED, "fused tcgen05 generation needs the discrete head width to be 0 or S");
    TcParams p{};
    p.image = static_cast<const uint8_t*>(m->tc_image);
    p.lay = make_layout(m->dims);
    p.x = x; p.k = k; p.mask = mask;
    p.step_tab = dev_table; p.temb = dev_table + (size_t)n_steps * 4; p.temb_stride = 0;
    p.n_steps = n_steps; p.dt = dt; p.u_jump = u_jump; p.seed = seed; p.jet_offset = jet_offset;
    p.B = B; p.N = N;
    tc_time_vectors_kernel<<<n_steps, 16 * (2 + 2 * kMaxL), 0, stream>>>(p.image, p.lay, p.temb, scratch);
    if (int rc = cuda_ok(cudaGetLastError(), "tc_time_vectors launch")) return rc;
    p.tvec = scratch;
    // bin the jets, every call: big ones get a tile each, small ones share tiles in pairs.  Where a jet runs (paired tile or
    // not, which rotation) depends on the jet alone, so its result does not depend on the size or composition of the call
    const BinLayout bl(B);
    int32_t* base = reinterpret_cast<int32_t*>(scratch + (((size_t)n_steps * (2 + 2 * m->dims.num_blocks) * 16 + 3) & ~(size_t)3));
    uint8_t* flag = reinterpret_cast<uint8_t*>(base + bl.flag);
    tc_bin_count_kernel<<<bl.nblocks, kBinThreads, 0, stream>>>(mask, B, N, ((N & 15) == 0 && (reinterpret_cast<uintptr_t>(mask) & 15) == 0) ? 1 : 0,
                                                                flag, base + bl.block_small);
    tc_bin_scan_kernel<<<1, 32, 0, stream>>>(base + bl.block_small, bl.nblocks, B, base + bl.block_off, base + bl.counts);
    tc_bin_fill_kernel<<<bl.nblocks, kBinThreads, 0, stream>>>(flag, base + bl.block_off, B, base + bl.small_list, base + bl.big_list);
    if (int rc = cuda_ok(cudaGetLastError(), "tc_bin launch")) return rc;
    p.counts = base + bl.counts;
    p.small_list = base + bl.small_list;
    p.big_list = base + bl.big_list;
    return dispatch<true>(m->dims, p, stream);
}

}  // namespace mmb
