// epic_mma.cu — the EPiC generation loop as register-resident warp-level tensor-core chains (mma.sync m16n8k16), sm_100a.
//
// Why a second tensor-core engine next to epic_tc.cu (tcgen05): the default EPiC is a chain of K = N = 16 GEMMs.  On tcgen05
// every link of that chain is a round trip  st.shared A tile -> fence.proxy.async -> CTA barrier -> tcgen05.mma -> commit ->
// mbarrier wait -> tcgen05.ld  (~500 cycles, seven per solver step) and the per-jet global MLP runs on one warp while the
// others wait; ncu of the round-1 kernel: tensor pipe 12 %, issue slots 52 %, barrier stalls first.  With warp-level MMA the
// accumulator fragment of one layer IS the A fragment of the next (row g / g+8, column pairs 2t, 2t+1 in both layouts), so a
// warp carries its particles through the whole network without leaving its registers:
//
//   * warp = up to 64 consecutive particles of ONE jet = one to four m16 tiles (four compile-time copies of the step loop;
//     a warp runs the copy that covers its last live particle).  86 % of JetClass-like jets fit one warp: no barrier, no
//     exchange, the per-jet work is done once.  Wider jets span ceil(rows / 64) warps of one CTA;
//   * per-particle Linear = 2 mma.sync per m-tile (two n8 tiles, K = 16), weights as pre-swizzled B fragments in shared
//     memory (one 8-byte load per lane per tile, shared by all m-tiles); bias = the C operand (pre-duplicated quads, no
//     moves); leaky-ReLU / residual / skip on the fp32 accumulator; pack to fp16 pairs = next A fragment;
//   * masked sum pooling: fp32 column sums over the thread's rows (mask as multiplier), then a three-stage xor butterfly
//     over the row groups — every lane ends with the sums of ITS fragment columns, which is an A fragment with identical rows;
//   * so the per-jet global MLP is tensor-core work too (M = 16, K = 16..48, N = 16) and stays in the fragment layout; the
//     per-jet bias of fc_local1 comes out as exactly the C operand the per-particle GEMM needs.  Jets that span several warps
//     exchange 16 partial sums through shared memory (named barrier per jet, ping-pong buffers) and each warp then runs the
//     same global MLP — identical bits in every warp;
//   * the hybrid update runs in the "owner" layout (lane = particle, two particles per lane for 3-4 tiles): logits / velocity
//     go through a per-warp staging tile, the first A fragment comes back through the same tile with ldmatrix.
//
// Operands: fp16 (11-bit mantissa, 8x finer than bf16; pooled sums enter scaled by 2^-7 against weights scaled by 2^7 — exact,
// and nothing can overflow), fp32 accumulate, fp32 residual stream / skip / pooling / update.
// Measured on B200 (tools/micro/hmma_rate.cu): HMMA.16816 latency 21 cycles, one per 8 cycles per scheduler (540 TFLOP/s);
// this kernel is bound by issue slots, not by the tensor pipe — every design choice above removes instructions.
//
// Reference semantics: SURVEY.md §A.2 (mp/models/architectures/epic.py:136-241, utils.py:112-172,
// mp/models/generative/multimodal_bridge_matching.py:90-113,199-216, bridges.py:38-45,106-132,179-201).
#include <cuda_fp16.h>

#include <type_traits>
#include <vector>

#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {
namespace {

constexpr int kH = 16;          // hidden width this engine is built for
// warps per CTA; the grid is persistent: kMinBlocks CTAs per SM.  Measured at C2 / dense: 8 warps x 2 CTAs per SM 4.07 / 1.98 M
// jets/s, 16 x 1: 3.93 / 1.73
constexpr int kW = 8;
constexpr int kMinBlocks = 2;
constexpr int kRowsPerWarp = 64;
constexpr int kMaxCls = 4;      // a jet spans at most this many warps (N <= 256)
constexpr int kKeys = 4 * kMaxCls;   // work lists: key = 4 (cls - 1) + (m-tiles of the jet's last warp - 1)
constexpr int kMaxL = 4;
constexpr int kCounterInts = 2 * kKeys;   // counts [kKeys] | cursors [kKeys]
constexpr int kStageBytes = 3072;   // per warp: A tile [64 rows][48 B]  /  logits [64][8] f32 + velocity [64][4] f32
constexpr int kSkipBytes = 4096;    // per warp: fp32 skip connection, [8][32 lanes] float4
constexpr int kPoolFloats = 32;     // per warp: two (ping-pong) slots of 16 partial column sums
constexpr float kSumScale = 1.0f / 128.0f;   // pooled sums enter the fp16 GEMMs scaled by 2^-7 (weights by 2^7)

// ---- image: B-fragment tiles (256 B each: lane l holds {b0, b1}) then bias quads (float4 per (vector, n-tile, t)) ----------------------
// Tile order (GT = ceil(G / 16)):  local_0 [2] | g0 [mean n0 n1 | sum n0 n1] | g1 [2] | g2 [2 GT] |
//   L x { fc_global1 [mean 2 | sum 2 | xg 2 GT] | fc_global2 [2 GT] | fc_local1 per-jet part [2 GT] | fc_local1 [2] | fc_local2 [2] } |
//   output [z n-tile, v n-tile] | head2 [1]
// Bias vectors (8 float4 each = [n-tile j][t] {b[8j+2t], b[8j+2t+1], b[8j+2t], b[8j+2t+1]}):
//   g1 | g2 [GT] | L x { fc_global2 [GT] | fc_local2 } | output | head2
template <int GT>
struct Lay {
    static constexpr int t_local0 = 0, t_g0 = 2, t_g1 = 6, t_g2 = 8, t_layer0 = 8 + 2 * GT;
    static constexpr int o_g1 = 0, o_g2 = 4 + 2 * GT, o_l1g = 4 + 4 * GT, o_l1 = 4 + 6 * GT, o_l2 = 6 + 6 * GT, layer_tiles = 8 + 6 * GT;
    static constexpr int v_g1 = 0, v_g2 = 1, v_layer0 = 1 + GT, ov_g2 = 0, ov_l2 = GT, layer_vecs = GT + 1;
    __host__ __device__ static constexpr int n_tiles(int L) { return t_layer0 + L * layer_tiles + 3; }
    __host__ __device__ static constexpr int n_vecs(int L) { return v_layer0 + L * layer_vecs + 2; }
    __host__ __device__ static constexpr size_t image_bytes(int L) { return (size_t)n_tiles(L) * 256 + (size_t)n_vecs(L) * 128; }
};

// ---- small PTX wrappers ---------------------------------------------------------------------------------------------------------------
// D = A * B + C (m16n8k16, fp16 in, fp32 accumulate); D and C are separate registers, so a shared bias quad needs no copy
__device__ __forceinline__ void mma(float (&d)[4], const uint32_t (&a)[4], const uint2 b, const float4 c) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
        : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y), "f"(c.x), "f"(c.y), "f"(c.z), "f"(c.w));
}
__device__ __forceinline__ void mma_acc(float (&d)[4], const uint32_t (&a)[4], const uint2 b) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&a)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]) : "r"(addr));
}

__device__ __forceinline__ void lrelu4(float (&c)[4]) {
    float t0, t1, t2, t3;
    fmul2(t0, t1, c[0], c[1], 0.01f, 0.01f);
    fmul2(t2, t3, c[2], c[3], 0.01f, 0.01f);
    c[0] = fmaxf(c[0], t0); c[1] = fmaxf(c[1], t1); c[2] = fmaxf(c[2], t2); c[3] = fmaxf(c[3], t3);
}
__device__ __forceinline__ float selu_f(float a) {   // branch-free
    const float scale = 1.0507009873554804934193349852946f;
    const float alpha_scale = 1.0507009873554804934193349852946f * 1.6732632423543772848170429916717f;
    const float neg = fmaf(alpha_scale, ex2_fast(a * 1.4426950408889634f), -alpha_scale);
    return a > 0.0f ? scale * a : neg;
}

// Named barrier of team `team` of class `cls` (a team = cls consecutive warps).  Warps move from class to class on their own,
// so teams of different classes are alive at the same time and every (class, team) pair needs its own hardware barrier:
// ids 1 .. sum_{c=2..4} kW / c, which must stay below 16.
__host__ __device__ constexpr int team_barrier(int cls, int team) {
    int base = 1;
    for (int c = kMaxCls; c > cls; --c) base += kW / c;
    return base + team;
}
static_assert(team_barrier(2, kW / 2 - 1) <= 15, "too many warps per CTA for one named barrier per team");

struct MmaParams {
    const uint8_t* image;
    int L, skip;
    float* x;                // [B,N,Dc] in/out (device); HOSTIO: the OUTPUT buffer, page-locked host memory mapped into the device
    uint8_t* k;              // [B,N] in/out (device); unused with HOSTIO
    const uint8_t* mask;
    // HOSTIO (mmb_generate_host, direct mode): the kernel reads the source state of a jet straight from the caller's page-locked
    // host buffers when a warp claims the jet, and writes the final state straight back — int64 tokens as the reference holds
    // them — so the PCIe traffic of a jet hides under the solver steps of the others, with no staging copy and no slicing
    const float* x_in;       // [B,N,Dc] host
    const long long* k_in;   // [B,N] host, int64
    long long* k_out;        // [B,N] host, int64
    int* bad_tokens;         // device flag: a token of a live particle was outside [0, S)
    const float* step_tab;   // [n_steps][4] (bc, cc, sp, t)
    int n_steps;
    float dt;
    const float* u_jump;     // [n_steps, B, N] or null
    uint64_t seed, jet_offset;
    int B, N;
    const float4* tvec;      // [n_steps][2 + 2L][8] bias quads of the per-step time vectors (prologue kernel)
    const float4* cvec;      // [B][1 + 2L][8] quads of the per-jet context terms of global_0 / fc_global1 / fc_local1, or null
    const int32_t* counts;   // [kKeys]: jets per key (empty jets are finished by the prologue and appear in no list)
    int32_t* cursors;        // [kKeys]: next unclaimed jet of each key (teams of `cls` warps claim dynamically)
    const int32_t* lists;    // [kKeys][B]: jets of each key
    const int32_t* jet_cnt;  // [B] live particles
};

// A column vector in the fragment layout (v[j][b] = element 8 j + 2 t + b, the same in every row group) as an A operand whose
// rows 0-7 carry the vector; rows 8-15 are zero (their outputs are never read) unless `dup`, which makes all 16 rows equal
// so that the OUTPUT quad {c0, c1, c2, c3} = {y[2t], y[2t+1], y[2t], y[2t+1]} can serve as a C operand for 16 particle rows.
__device__ __forceinline__ void vec_frag(uint32_t (&a)[4], float v00, float v01, float v10, float v11, bool dup = false) {
    a[0] = pack_f16(v00, v01);
    a[2] = pack_f16(v10, v11);
    a[1] = dup ? a[0] : 0u;
    a[3] = dup ? a[2] : 0u;
}

template <int DC, int S, int SH, int GT, bool HOSTIO, bool CTX>
__global__ void __launch_bounds__(kW * 32, kMinBlocks) epic_mma_generate_kernel(const MmaParams p) {
    using LY = Lay<GT>;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int L = p.L;

    // ---- carve shared memory: image | per-warp staging tiles | per-warp skip buffers | pooling exchange
    const size_t image_bytes = LY::image_bytes(L);
    const uint2* tiles_lane = reinterpret_cast<const uint2*>(smem) + lane;                       // tile i of this lane: tiles_lane[32 i]
    const float4* quads_t = reinterpret_cast<const float4*>(smem + (size_t)LY::n_tiles(L) * 256) + t;   // quad (v, j): quads_t[8 v + 4 j]
    uint8_t* s_warp = smem + ((image_bytes + 127) & ~(size_t)127);
    uint8_t* stage = s_warp + warp * kStageBytes;
    float4* skipbuf = reinterpret_cast<float4*>(s_warp + kW * kStageBytes + warp * kSkipBytes) + lane;
    float* pool_all = reinterpret_cast<float*>(s_warp + kW * (kStageBytes + kSkipBytes));
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.image);
        uint4* dst = reinterpret_cast<uint4*>(smem);
        const int n16 = (int)(image_bytes / 16);
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    __syncthreads();

    __shared__ int s_claim[kW];
    const int N = p.N;
    const bool skip_on = p.skip != 0;
    auto tile = [&](int idx) { return tiles_lane[idx * 32]; };
    auto quad = [&](int vec, int j) { return quads_t[8 * vec + 4 * j]; };

    // One jet (or this warp's 64-row slice of it) through all solver steps.  `team` = index of the group of `cls` consecutive
    // warps that carries the jet: named barrier 1 + team, exchange buffers of the team's first warp onwards.
    auto process = [&](const int jet, const int cls, const int slice, const int team) {
    // the two particles this lane OWNS (state, update): rows lane and lane + 32 of the warp's slice
    const int n0 = kRowsPerWarp * slice + lane, n1 = n0 + 32;
    const size_t jbase = (size_t)jet * N;
    const bool live0 = n0 < N && p.mask[jbase + n0] != 0, live1 = n1 < N && p.mask[jbase + n1] != 0;
    const unsigned bal0 = __ballot_sync(0xffffffffu, live0), bal1 = __ballot_sync(0xffffffffu, live1);
    const float inv_cnt = 1.0f / (float)__ldg(p.jet_cnt + jet);
    const int bar_id = team_barrier(cls, team), bar_threads = 32 * cls;
    float* pool_mine = pool_all + warp * kPoolFloats;
    const float* pool_jet = pool_all + (team * cls) * kPoolFloats;
    const uint64_t jet_key = p.jet_offset + (uint64_t)jet;

    auto run = [&](auto nmt_tag) {
        constexpr int NMT = decltype(nmt_tag)::value;
        constexpr bool TWO = NMT > 2;   // this lane owns a second particle
        float xs0[DC], xs1[DC];
        int kk0 = 0, kk1 = 0;
        // Features of the slice: rows are 12 B apart, so per-lane scalar accesses touch every 32-byte sector three times —
        // harmless in HBM, a 3x cost over PCIe (direct mode).  With N % 4 == 0 the rows of a slice form whole 16-byte chunks:
        // the warp moves them as float4 through the staging tile.
        const bool vec_io = (N & 3) == 0;
        const float* xin = HOSTIO ? p.x_in : p.x;
        if (vec_io) {
            const int rows = min(16 * NMT, N - kRowsPerWarp * slice);
            const float4* src = reinterpret_cast<const float4*>(xin + (jbase + (size_t)kRowsPerWarp * slice) * DC);
            for (int i = lane; i < rows * DC / 4; i += 32) reinterpret_cast<float4*>(stage)[i] = __ldg(src + i);
            __syncwarp();
            const float* st = reinterpret_cast<const float*>(stage);
#pragma unroll
            for (int c = 0; c < DC; ++c) {
                xs0[c] = live0 ? st[lane * DC + c] : 0.0f;
                xs1[c] = (TWO && live1) ? st[(lane + 32) * DC + c] : 0.0f;
            }
            __syncwarp();
        } else {
#pragma unroll
            for (int c = 0; c < DC; ++c) {
                xs0[c] = live0 ? xin[(jbase + n0) * DC + c] : 0.0f;
                xs1[c] = (TWO && live1) ? xin[(jbase + n1) * DC + c] : 0.0f;
            }
        }
        if constexpr (HOSTIO) {
            const long long q0 = live0 ? p.k_in[jbase + n0] : 0, q1 = (TWO && live1) ? p.k_in[jbase + n1] : 0;
            if (q0 < 0 || q0 >= S || q1 < 0 || q1 >= S) atomicOr(p.bad_tokens, 1);   // the reference asserts (bridges.py:111-115)
            kk0 = (int)q0 & (S - 1);
            kk1 = (int)q1 & (S - 1);
        } else {
            if (live0) kk0 = p.k[jbase + n0];
            if (TWO && live1) kk1 = p.k[jbase + n1];
        }
        // row masks of this thread's fragment rows, as multipliers of the pooling sums: [mt][hh] = row 16 mt + 8 hh + g
        float mk[NMT][2];
#pragma unroll
        for (int mt = 0; mt < NMT; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
                mk[mt][hh] = (((mt < 2 ? bal0 : bal1) >> (16 * (mt & 1) + 8 * hh + g)) & 1u) ? 1.0f : 0.0f;
        float xl[NMT][2][4];
        uint32_t af[NMT][4];
        uint32_t uq[TWO ? 8 : 4] = {};
        int pp = 0;   // ping-pong slot of the pooling exchange

        auto pack_rows = [&](uint32_t (&a)[NMT][4], const float (&v)[NMT][2][4]) {
#pragma unroll
            for (int mt = 0; mt < NMT; ++mt) {
                a[mt][0] = pack_f16(v[mt][0][0], v[mt][0][1]);
                a[mt][1] = pack_f16(v[mt][0][2], v[mt][0][3]);
                a[mt][2] = pack_f16(v[mt][1][0], v[mt][1][1]);
                a[mt][3] = pack_f16(v[mt][1][2], v[mt][1][3]);
            }
        };
        // masked column sums of xl over the jet: this warp's rows by multiply-adds + xor butterfly, then the jet's other warps
        auto pool = [&](float (&s)[2][2]) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                float a0, a1;
                fmul2(a0, a1, xl[0][j][0], xl[0][j][1], mk[0][0], mk[0][0]);
                ffma2(a0, a1, xl[0][j][2], xl[0][j][3], mk[0][1], mk[0][1], a0, a1);
#pragma unroll
                for (int mt = 1; mt < NMT; ++mt) {
                    ffma2(a0, a1, xl[mt][j][0], xl[mt][j][1], mk[mt][0], mk[mt][0], a0, a1);
                    ffma2(a0, a1, xl[mt][j][2], xl[mt][j][3], mk[mt][1], mk[mt][1], a0, a1);
                }
                s[j][0] = a0; s[j][1] = a1;
            }
#pragma unroll
            for (int off = 4; off <= 16; off <<= 1) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    s[j][0] += __shfl_xor_sync(0xffffffffu, s[j][0], off);
                    s[j][1] += __shfl_xor_sync(0xffffffffu, s[j][1], off);
                }
            }
            if (cls > 1) {
                if (g == 0) *reinterpret_cast<float4*>(pool_mine + pp * 16 + 4 * t) = make_float4(s[0][0], s[0][1], s[1][0], s[1][1]);
                named_bar(bar_id, bar_threads);
                float4 acc = *reinterpret_cast<const float4*>(pool_jet + pp * 16 + 4 * t);
                for (int w = 1; w < cls; ++w) {
                    const float4 q = *reinterpret_cast<const float4*>(pool_jet + w * kPoolFloats + pp * 16 + 4 * t);
                    acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
                }
                s[0][0] = acc.x; s[0][1] = acc.y; s[1][0] = acc.z; s[1][1] = acc.w;
                pp ^= 1;
            }
        };

        for (int step = 0; step < p.n_steps; ++step) {
            const float4* tvq = p.tvec + (size_t)step * (2 + 2 * L) * 8 + t;   // quad (v, j): tvq[8 v + 4 j]
            // time vector v (>= 1) plus the jet's context term of the same Linear (the reference's context = [t_emb | ctx])
            auto ctx_quad = [&](int v, int j) {
                float4 b = __ldg(tvq + 8 * v + 4 * j);
                if constexpr (CTX) {
                    const float4 c = __ldg(p.cvec + ((size_t)jet * (1 + 2 * L) + (v - 1)) * 8 + 4 * j + t);
                    b.x += c.x; b.y += c.y; b.z += c.z; b.w += c.w;
                }
                return b;
            };
            // ---- (a) first A tile: [x_hi, x_lo, onehot(k)] per particle through the staging tile; every lane writes its rows
            // every step (dead rows: zeros — the tile doubles as the logits staging area)
            {
                static_assert(DC == 3, "row packing below is written for three continuous features");
                auto put_row = [&](int row, const float (&xs)[DC], int kk, bool live) {
                    float hi[DC], lo[DC];
#pragma unroll
                    for (int c = 0; c < DC; ++c) {
                        hi[c] = __half2float(__float2half_rn(xs[c]));
                        lo[c] = xs[c] - hi[c];
                    }
                    const uint32_t sel = live ? (0x3C00u << (16 * (kk & 1))) : 0u;
                    const int kw = kk >> 1;
                    uint32_t w[8];
                    w[0] = pack_f16(hi[0], hi[1]);     // xs == 0 on dead rows
                    w[1] = pack_f16(hi[2], lo[0]);
                    w[2] = pack_f16(lo[1], lo[2]);
#pragma unroll
                    for (int i = 0; i < 4; ++i) w[3 + i] = (i < S / 2 && kw == i) ? sel : 0u;
                    w[7] = 0u;
                    *reinterpret_cast<uint4*>(stage + row * 48) = make_uint4(w[0], w[1], w[2], w[3]);
                    *reinterpret_cast<uint4*>(stage + row * 48 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
                };
                put_row(lane, xs0, kk0, live0);
                if constexpr (TWO) put_row(lane + 32, xs1, kk1, live1);
            }
            __syncwarp();
#pragma unroll
            for (int mt = 0; mt < NMT; ++mt)
                ldmatrix_x4(af[mt], smem_u32(stage + (16 * mt + (lane & 7) + 8 * ((lane >> 3) & 1)) * 48 + (lane >> 4) * 16));

            // ---- (b) local_0 (+ folded embeddings), leaky-ReLU -> xl; skip copy.  Dead rows carry finite junk from here on:
            // rows never mix except in the pooling sums, which multiply by the mask.
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const float4 b = __ldg(tvq + 4 * j);
                const uint2 w = tile(LY::t_local0 + j);
#pragma unroll
                for (int mt = 0; mt < NMT; ++mt) {
                    mma(xl[mt][j], af[mt], w, b);
                    lrelu4(xl[mt][j]);
                    if (skip_on) skipbuf[(2 * mt + j) * 32] = make_float4(xl[mt][j][0], xl[mt][j][1], xl[mt][j][2], xl[mt][j][3]);
                }
            }
            pack_rows(af, xl);
            // ---- (c) pooling + EPiC_Projection globals (epic.py:187-190); per-jet vectors live as xg[j][b] = element 8 j + 2 t + b
            float ps[2][2];
            pool(ps);
            float xg[2 * GT][2], skg[2 * GT][2];
            {
                uint32_t a_mean[4], a_sum[4], a[4];
                vec_frag(a_mean, ps[0][0] * inv_cnt, ps[0][1] * inv_cnt, ps[1][0] * inv_cnt, ps[1][1] * inv_cnt);
                vec_frag(a_sum, ps[0][0] * kSumScale, ps[0][1] * kSumScale, ps[1][0] * kSumScale, ps[1][1] * kSumScale);
                float c[2][4];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    mma(c[j], a_mean, tile(LY::t_g0 + j), ctx_quad(1, j));
                    mma_acc(c[j], a_sum, tile(LY::t_g0 + 2 + j));
                }
                vec_frag(a, lrelu_fast(c[0][0]), lrelu_fast(c[0][1]), lrelu_fast(c[1][0]), lrelu_fast(c[1][1]));
#pragma unroll
                for (int j = 0; j < 2; ++j) mma(c[j], a, tile(LY::t_g1 + j), quad(LY::v_g1, j));
                vec_frag(a, lrelu_fast(c[0][0]), lrelu_fast(c[0][1]), lrelu_fast(c[1][0]), lrelu_fast(c[1][1]));
#pragma unroll
                for (int j = 0; j < 2 * GT; ++j) {
                    float d[4];
                    mma(d, a, tile(LY::t_g2 + j), quad(LY::v_g2 + (j >> 1), j & 1));
                    xg[j][0] = lrelu_fast(d[0]); xg[j][1] = lrelu_fast(d[1]);
                    skg[j][0] = skip_on ? xg[j][0] : 0.0f; skg[j][1] = skip_on ? xg[j][1] : 0.0f;
                }
            }
            // ---- EPiC layers (epic.py:217-241, 152-155)
            for (int l = 0; l < L; ++l) {
                const uint2* tl = tiles_lane + (LY::t_layer0 + l * LY::layer_tiles) * 32;
                const float4* ql = quads_t + 8 * (LY::v_layer0 + l * LY::layer_vecs);
                if (l > 0) pool(ps);   // layer 0 pools the same tensor the projection pooled
                float4 bl1[2];
                {
                    uint32_t a_mean[4], a_sum[4], a[4];
                    vec_frag(a_mean, ps[0][0] * inv_cnt, ps[0][1] * inv_cnt, ps[1][0] * inv_cnt, ps[1][1] * inv_cnt);
                    vec_frag(a_sum, ps[0][0] * kSumScale, ps[0][1] * kSumScale, ps[1][0] * kSumScale, ps[1][1] * kSumScale);
                    float c[2][4];
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        mma(c[j], a_mean, tl[(LY::o_g1 + j) * 32], ctx_quad(2 + 2 * l, j));
                        mma_acc(c[j], a_sum, tl[(LY::o_g1 + 2 + j) * 32]);
                    }
#pragma unroll
                    for (int gt = 0; gt < GT; ++gt) {   // xg k-steps
                        vec_frag(a, xg[2 * gt][0], xg[2 * gt][1], xg[2 * gt + 1][0], xg[2 * gt + 1][1]);
#pragma unroll
                        for (int j = 0; j < 2; ++j) mma_acc(c[j], a, tl[(LY::o_g1 + 4 + 2 * gt + j) * 32]);
                    }
                    vec_frag(a, lrelu_fast(c[0][0]), lrelu_fast(c[0][1]), lrelu_fast(c[1][0]), lrelu_fast(c[1][1]));
                    // fc_global2 + residual (epic.py:231-232), trunk skip (epic.py:155)
                    float xm[2 * GT][2];
#pragma unroll
                    for (int j = 0; j < 2 * GT; ++j) {
                        float4 b = ql[8 * (LY::ov_g2 + (j >> 1)) + 4 * (j & 1)];
                        b.x += xg[j][0]; b.y += xg[j][1];
                        float d[4];
                        mma(d, a, tl[(LY::o_g2 + j) * 32], b);
                        xm[j][0] = lrelu_fast(d[0]); xm[j][1] = lrelu_fast(d[1]);
                        xg[j][0] = xm[j][0] + skg[j][0]; xg[j][1] = xm[j][1] + skg[j][1];
                    }
                    // per-jet part of fc_local1: time vector + Wl1[:, H:H+G] xg   (epic.py:233-238); all 16 rows equal, so the
                    // output quads are the C operand of the per-particle GEMM
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        float d[4];
                        vec_frag(a, xm[0][0], xm[0][1], xm[1][0], xm[1][1], true);
                        mma(d, a, tl[(LY::o_l1g + j) * 32], ctx_quad(3 + 2 * l, j));
#pragma unroll
                        for (int gt = 1; gt < GT; ++gt) {
                            vec_frag(a, xm[2 * gt][0], xm[2 * gt][1], xm[2 * gt + 1][0], xm[2 * gt + 1][1], true);
                            mma_acc(d, a, tl[(LY::o_l1g + 2 * gt + j) * 32]);
                        }
                        bl1[j] = make_float4(d[0], d[1], d[2], d[3]);
                    }
                }
                // fc_local1 -> leaky-ReLU -> fc_local2 + residual -> leaky-ReLU, trunk skip
                uint32_t a1[NMT][4];
                {
                    float acc[NMT][2][4];
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const uint2 w = tl[(LY::o_l1 + j) * 32];
#pragma unroll
                        for (int mt = 0; mt < NMT; ++mt) {
                            mma(acc[mt][j], af[mt], w, bl1[j]);
                            lrelu4(acc[mt][j]);
                        }
                    }
                    pack_rows(a1, acc);
                }
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const float4 b = ql[8 * LY::ov_l2 + 4 * j];
                    const uint2 w = tl[(LY::o_l2 + j) * 32];
#pragma unroll
                    for (int mt = 0; mt < NMT; ++mt) {
                        float4 c;
                        fadd2(c.x, c.y, xl[mt][j][0], xl[mt][j][1], b.x, b.y);
                        fadd2(c.z, c.w, xl[mt][j][2], xl[mt][j][3], b.x, b.y);
                        mma(xl[mt][j], a1[mt], w, c);
                        lrelu4(xl[mt][j]);
                        if (skip_on) {
                            const float4 sk = skipbuf[(2 * mt + j) * 32];
                            fadd2(xl[mt][j][0], xl[mt][j][1], xl[mt][j][0], xl[mt][j][1], sk.x, sk.y);
                            fadd2(xl[mt][j][2], xl[mt][j][3], xl[mt][j][2], xl[mt][j][3], sk.z, sk.w);
                        }
                    }
                }
                pack_rows(af, xl);
            }
            // ---- output layer (+ head Linear 0 folded in), SELU, head Linear 2   (epic.py:158-162, mbm.py:105-111)
            __syncwarp();   // every lane is past its ldmatrix of this step: the staging tile may be overwritten
            {
                const uint2* tt = tiles_lane + (LY::t_layer0 + L * LY::layer_tiles) * 32;
                const float4* qt = quads_t + 8 * (LY::v_layer0 + L * LY::layer_vecs);
                [[maybe_unused]] const float4 bz = qt[0], bv = qt[4], b2 = qt[8];
                [[maybe_unused]] const uint2 wz = tt[0], wv = tt[32], w2 = tt[64];
                float* slog = reinterpret_cast<float*>(stage);
                float* sv = reinterpret_cast<float*>(stage + 2048);
#pragma unroll
                for (int mt = 0; mt < NMT; ++mt) {
                    float hz[4], hv[4];
                    mma(hz, af[mt], wz, bz);
                    mma(hv, af[mt], wv, bv);
                    if constexpr (SH > 0) {
                        uint32_t az[4];
                        az[0] = pack_f16(selu_f(hz[0]), selu_f(hz[1]));
                        az[1] = pack_f16(selu_f(hz[2]), selu_f(hz[3]));
                        az[2] = az[3] = 0u;
                        mma(hz, az, w2, b2);
                    }
                    // fragment layout -> owner layout through the staging tile
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int row = 16 * mt + 8 * hh + g;
                        *reinterpret_cast<float2*>(slog + row * 8 + 2 * t) = make_float2(hz[2 * hh], hz[2 * hh + 1]);
                        if (t < 2) *reinterpret_cast<float2*>(sv + row * 4 + 2 * t) = make_float2(hv[2 * hh], hv[2 * hh + 1]);
                    }
                }
            }
            __syncwarp();
            // ---- hybrid update of the owned particles (bridges.py:38-45,179-201)
            if (!p.u_jump && (step & 3) == 0) {   // one Philox block serves four particles x one step: share it inside the lane quad
#pragma unroll
                for (int q = 0; q < (TWO ? 2 : 1); ++q) {
                    const int n = q ? n1 : n0;
                    const uint4 blk = philox_block(p.seed, jet_key, 0, step + (n & 3), n >> 2);
                    uint32_t a0 = blk.x, a1 = blk.y, a2 = blk.z, a3 = blk.w;
                    {
                        const bool hi = (lane & 2) != 0;
                        const uint32_t r0 = __shfl_xor_sync(0xffffffffu, hi ? a0 : a2, 2), r1 = __shfl_xor_sync(0xffffffffu, hi ? a1 : a3, 2);
                        if (hi) { a0 = r0; a1 = r1; } else { a2 = r0; a3 = r1; }
                    }
                    {
                        const bool hi = (lane & 1) != 0;
                        const uint32_t r0 = __shfl_xor_sync(0xffffffffu, hi ? a0 : a1, 1), r1 = __shfl_xor_sync(0xffffffffu, hi ? a2 : a3, 1);
                        if (hi) { a0 = r0; a2 = r1; } else { a1 = r0; a3 = r1; }
                    }
                    uq[4 * q + 0] = a0; uq[4 * q + 1] = a1; uq[4 * q + 2] = a2; uq[4 * q + 3] = a3;
                }
            }
            {
                const float bc = __ldg(p.step_tab + step * 4 + 0), cc = __ldg(p.step_tab + step * 4 + 1);
                const int ph = step & 3;
                auto update = [&](int row, int n, float (&xs)[DC], int& kk, bool live, uint32_t ubits) {
                    if (!live) return;
                    const float4 v4 = *reinterpret_cast<const float4*>(stage + 2048 + row * 16);
                    const float4 l0 = *reinterpret_cast<const float4*>(stage + row * 32);
                    float lg[S];
                    lg[0] = l0.x; lg[1] = l0.y; lg[2] = l0.z; lg[3] = l0.w;
                    if constexpr (S > 4) {
                        const float4 l1 = *reinterpret_cast<const float4*>(stage + row * 32 + 16);
                        lg[4] = l1.x; lg[5] = l1.y; lg[6] = l1.z; lg[7] = l1.w;
                    }
                    xs[0] = fmaf(p.dt, v4.x, xs[0]); xs[1] = fmaf(p.dt, v4.y, xs[1]); xs[2] = fmaf(p.dt, v4.z, xs[2]);
                    const float u = p.u_jump ? __ldg(p.u_jump + ((size_t)step * p.B + jet) * N + n) : u01(ubits);
                    kk = telegraph_jump_fast_ex2<S>(lg, kk, u, p.dt, bc, cc);
                };
                update(lane, n0, xs0, kk0, live0, ph == 0 ? uq[0] : ph == 1 ? uq[1] : ph == 2 ? uq[2] : uq[3]);
                if constexpr (TWO) update(lane + 32, n1, xs1, kk1, live1, ph == 0 ? uq[4] : ph == 1 ? uq[5] : ph == 2 ? uq[6] : uq[7]);
            }
            __syncwarp();   // the staging tile becomes the A tile of the next step
        }
        // ---- final state: live particles as computed, dead ones 0 (x * mask, k * mask)
        if (vec_io) {
            float* st = reinterpret_cast<float*>(stage);
#pragma unroll
            for (int c = 0; c < DC; ++c) {
                st[lane * DC + c] = live0 ? xs0[c] : 0.0f;
                st[(lane + 32) * DC + c] = (TWO && live1) ? xs1[c] : 0.0f;
            }
            __syncwarp();
            const int rows = min(kRowsPerWarp, N - kRowsPerWarp * slice);
            float4* dst = reinterpret_cast<float4*>(p.x + (jbase + (size_t)kRowsPerWarp * slice) * DC);
            for (int i = lane; i < rows * DC / 4; i += 32) dst[i] = reinterpret_cast<const float4*>(stage)[i];
            __syncwarp();
        } else {
            if (n0 < N)
#pragma unroll
                for (int c = 0; c < DC; ++c) p.x[(jbase + n0) * DC + c] = live0 ? xs0[c] : 0.0f;
            if (n1 < N)   // NMT <= 2: rows 32-63 of the slice are dead
#pragma unroll
                for (int c = 0; c < DC; ++c) p.x[(jbase + n1) * DC + c] = (TWO && live1) ? xs1[c] : 0.0f;
        }
        if (n0 < N) {
            if constexpr (HOSTIO) p.k_out[jbase + n0] = live0 ? kk0 : 0;
            else p.k[jbase + n0] = (uint8_t)(live0 ? kk0 : 0);
        }
        if (n1 < N) {
            if constexpr (HOSTIO) p.k_out[jbase + n1] = (TWO && live1) ? kk1 : 0;
            else p.k[jbase + n1] = (uint8_t)((TWO && live1) ? kk1 : 0);
        }
        // rows past the last live particle have no warp: the team zeroes them
        const int tail0 = kRowsPerWarp * cls;
        if (vec_io) {
            float4* dst = reinterpret_cast<float4*>(p.x + (jbase + (size_t)tail0) * DC);
            for (int i = 32 * slice + lane; i < (N - tail0) * DC / 4; i += 32 * cls) dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int m = tail0 + 32 * slice + lane; m < N; m += 32 * cls) {
            if (!vec_io)
#pragma unroll
                for (int c = 0; c < DC; ++c) p.x[(jbase + m) * DC + c] = 0.0f;
            if constexpr (HOSTIO) p.k_out[jbase + m] = 0;
            else p.k[jbase + m] = 0;
        }
    };
    if ((bal1 >> 16) != 0u) run(std::integral_constant<int, 4>{});
    else if (bal1 != 0u) run(std::integral_constant<int, 3>{});
    else if ((bal0 >> 16) != 0u) run(std::integral_constant<int, 2>{});
    else run(std::integral_constant<int, 1>{});
    };

    // ---- persistent scheduling.  Jets wait in lists keyed by (warps they span, m-tiles of their last warp); a team of `cls`
    // consecutive warps claims the next jet of a key with one atomic (single-warp jets, the bulk, warp by warp).  The whole chip
    // walks the keys widest-first, so that (a) the longest jobs start first (LPT) and (b) at any moment the warps of the chip
    // work on neighbours in the list, i.e. run the same copy of the step loop.
    // Two alternatives were measured with per-job records (profiles/r02_mma_timeline.md) and removed: every SM starting on its
    // own key made no job faster and ended less evenly, and time slicing small calls cost more in warps waiting for the previous
    // slice of a jet than the shorter tail gave back (4096 jets: 1.35 ms against 0.94 ms unsliced).
    for (int visit = 0; visit < kKeys; ++visit) {
        const int key = kKeys - 1 - visit;
        const int n_key = __ldg(p.counts + key);
        if (n_key == 0) continue;
        const int cls = key / 4 + 1;
        const int team = warp / cls, slice = warp - team * cls;
        if ((team + 1) * cls > kW) continue;           // warps left over when cls does not divide kW sit this key out
        int32_t* cursor = p.cursors + key;
        for (;;) {
            int idx = 0;
            if (slice == 0) {
                if (lane == 0) idx = atomicAdd(cursor, 1);
                idx = __shfl_sync(0xffffffffu, idx, 0);
                if (cls > 1 && lane == 0) s_claim[team * cls] = idx;
            }
            if (cls > 1) {
                named_bar(team_barrier(cls, team), 32 * cls);
                idx = s_claim[team * cls];
                named_bar(team_barrier(cls, team), 32 * cls);   // everyone has read the claim before the leader overwrites it
            }
            if (idx >= n_key) break;
            const int jet = __ldg(p.lists + (size_t)key * p.B + idx);
            process(jet, cls, slice, team);
        }
    }
}

// ---- prologue: per-step time vectors + binning of the jets by the number of warps they span ---------------------------------------------
// blocks [0, n_steps): vectors of one step, from the fp32 weights (same for every jet), written as C-operand quads:
//   v0 = local_0 bias + W0[:, T:T+C] a + W0[:, :T] temb      (a = bias of the continuous embedding)
//   v1 = global_0 bias + G0[:, 2H:] temb;  per layer: fc_global1 bias + time part, fc_local1 bias + time part
// blocks [n_steps, ...): one thread per jet: live count, last live index -> key (warps spanned, m-tiles of the last warp); jets
// of a key are appended to its list (order irrelevant: a jet's result does not depend on where or when it runs).  Empty jets get the reference's result right here:
// the mean pool divides by zero (epic.py:141), every feature becomes NaN, tokens are multiplied by the mask -> 0.
constexpr int kPrologueThreads = 256;
__global__ void __launch_bounds__(kPrologueThreads) mma_prologue_kernel(const float* __restrict__ W, MmbEpicLayout Lo, MmbEpicDims d,
                                                                        const float* __restrict__ temb, int n_steps, float4* __restrict__ tvec,
                                                                        const float* __restrict__ context, float4* __restrict__ cvec, int ctx_blocks,
                                                                        const uint8_t* __restrict__ mask, int B, int N, int32_t* __restrict__ counts,
                                                                        int32_t* __restrict__ lists, int32_t* __restrict__ jet_cnt,
                                                                        float* __restrict__ x, uint8_t* __restrict__ k, long long* __restrict__ k64) {
    const int T = d.dim_time_emb, C = d.dim_cont_emb, D = d.dim_disc_emb, H = d.dim_hidden_local, G = d.dim_hidden_glob, L = d.num_blocks,
              X = d.dim_context, TX = T + X;
    // the context-consuming Linear `v` (1: global_0; 2 + 2l: fc_global1; 3 + 2l: fc_local1), output o: bias and its [time | context] columns
    auto ctx_columns = [&](int v, int o, float& bias) -> const float* {
        if (v == 1) { bias = W[Lo.global0_b + o]; return W + Lo.global0_w + (size_t)o * (2 * H + TX) + 2 * H; }
        const float* Wl = W + Lo.layer0 + (size_t)((v - 2) >> 1) * Lo.layer_stride;
        if (v & 1) { bias = Wl[Lo.l_l1_b + o]; return Wl + Lo.l_l1_w + (size_t)o * (H + G + TX) + H + G; }
        bias = Wl[Lo.l_g1_b + o];
        return Wl + Lo.l_g1_w + (size_t)o * (2 * H + G + TX) + 2 * H + G;
    };
    if ((int)blockIdx.x >= n_steps && (int)blockIdx.x < n_steps + ctx_blocks) {
        // one thread per (jet, Linear, quad): W[:, T:T+X] ctx_jet for two outputs, in the C-operand quad layout of the time vectors
        const size_t idx = (size_t)((int)blockIdx.x - n_steps) * kPrologueThreads + threadIdx.x;
        const int q = (int)(idx & 7), v = (int)((idx >> 3) % (size_t)(1 + 2 * L)) + 1;
        const size_t jet = (idx >> 3) / (size_t)(1 + 2 * L);
        if (jet < (size_t)B) {
            const int j = q >> 2, t = q & 3;
            const float* cj = context + jet * X;
            float unused, b[2];
            for (int e = 0; e < 2; ++e) {
                const float* wt = ctx_columns(v, 8 * j + 2 * t + e, unused) + T;
                float acc = 0.0f;
                for (int i = 0; i < X; ++i) acc = fmaf(wt[i], cj[i], acc);
                b[e] = acc;
            }
            cvec[idx] = make_float4(b[0], b[1], b[0], b[1]);
        }
        return;
    }
    const int bin_block0 = n_steps + ctx_blocks;
    if ((int)blockIdx.x < n_steps) {
        __shared__ float s_vec[2 + 2 * kMaxL][16];
        const int step = blockIdx.x, v = threadIdx.x >> 4, o = threadIdx.x & 15;
        if (v < 2 + 2 * L) {
            const float* te = temb + (size_t)step * T;
            float acc;
            const float* wt;
            if (v == 0) {
                const float* w0 = W + Lo.local0_w + (size_t)o * (T + C + D);
                acc = W[Lo.local0_b + o];
                for (int c = 0; c < C; ++c) acc = fmaf(w0[T + c], W[Lo.emb_cont_b + c], acc);
                wt = w0;
            } else {
                wt = ctx_columns(v, o, acc);
            }
            for (int i = 0; i < T; ++i) acc = fmaf(wt[i], te[i], acc);
            s_vec[v][o] = acc;
        }
        __syncthreads();
        if (v < 2 + 2 * L && o < 8) {   // quad (j, t) = {b[8j+2t], b[8j+2t+1], same, same}
            const int j = o >> 2, t = o & 3;
            const float b0 = s_vec[v][8 * j + 2 * t], b1 = s_vec[v][8 * j + 2 * t + 1];
            tvec[((size_t)step * (2 + 2 * L) + v) * 8 + 4 * j + t] = make_float4(b0, b1, b0, b1);
        }
        return;
    }
    __shared__ int s_cnt[kKeys], s_base[kKeys];
    if (threadIdx.x < kKeys) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int jet = ((int)blockIdx.x - bin_block0) * kPrologueThreads + threadIdx.x;
    int cls = -1, key = 0, pos = 0;
    if (jet < B) {
        const uint8_t* row = mask + (size_t)jet * N;
        int cnt = 0, last = 0;
        if ((N & 15) == 0 && (reinterpret_cast<uintptr_t>(mask) & 15) == 0) {
            for (int i = 0; i < N; i += 16) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(row + i));
                const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int b = 0; b < 4; ++b)
                        if ((w[j] >> (8 * b)) & 0xffu) { ++cnt; last = i + 4 * j + b + 1; }
            }
        } else {
            for (int i = 0; i < N; ++i)
                if (row[i]) { ++cnt; last = i + 1; }
        }
        jet_cnt[jet] = cnt;
        cls = (last + kRowsPerWarp - 1) / kRowsPerWarp;
        if (cls > 0) {
            key = 4 * (cls - 1) + (last - kRowsPerWarp * (cls - 1) + 15) / 16 - 1;   // m-tiles of the jet's last warp
            pos = atomicAdd(&s_cnt[key], 1);
        }
    }
    __syncthreads();
    if (threadIdx.x < kKeys) s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]) : 0;
    __syncthreads();
    if (cls > 0) lists[(size_t)key * B + s_base[key] + pos] = jet;
    if (cls == 0) {
        const float nan = __int_as_float(0x7fc00000);
        for (int i = 0; i < N * d.dim_continuous; ++i) x[(size_t)jet * N * d.dim_continuous + i] = nan;
        if (k64) for (int i = 0; i < N; ++i) k64[(size_t)jet * N + i] = 0;
        else for (int i = 0; i < N; ++i) k[(size_t)jet * N + i] = 0;
    }
}

inline uint16_t to_f16(float v) { __half h = __float2half_rn(v); return *reinterpret_cast<uint16_t*>(&h); }

// One k16 x n8 B-fragment tile of y = W x: lane (g, t) holds W[n0 + g][k0 + 2t, +1] and W[n0 + g][k0 + 2t + 8, +9];
// `w(o, k)` returns the (already folded) weight or 0 outside the matrix.
template <typename F>
void fill_tile(std::vector<uint16_t>& img, int idx, int n0, int k0, F w) {
    for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, t = lane & 3;
        for (int e = 0; e < 4; ++e) img[((size_t)idx * 32 + lane) * 4 + e] = to_f16((float)w(n0 + g, k0 + 2 * t + (e & 1) + 8 * (e >> 1)));
    }
}
// bias vector `vec` (8 float4): quad (j, t) = {b[8j+2t], b[8j+2t+1], same, same}
template <typename F>
void fill_vec(std::vector<float>& q, int vec, F b) {
    for (int j = 0; j < 2; ++j)
        for (int t = 0; t < 4; ++t) {
            float* o = q.data() + ((size_t)vec * 8 + 4 * j + t) * 4;
            o[0] = o[2] = b(8 * j + 2 * t);
            o[1] = o[3] = b(8 * j + 2 * t + 1);
        }
}

template <int GT>
int build_image_gt(const MmbEpicDims& d, const MmbEpicLayout& Lo, const float* W, void** out, size_t* out_bytes) {
    using LY = Lay<GT>;
    const int Dc = d.dim_continuous, S = d.vocab_size, T = d.dim_time_emb, C = d.dim_cont_emb, D = d.dim_disc_emb, H = kH,
              G = d.dim_hidden_glob, L = d.num_blocks, Sh = d.disc_head_hidden;
    const int K0 = T + C + D, TX = T + d.dim_context;   // context-consuming Linears: [... | time T | context X] columns
    std::vector<uint16_t> img((size_t)LY::n_tiles(L) * 128, 0);
    std::vector<float> quads((size_t)LY::n_vecs(L) * 32, 0.0f);
    const double inv_scale = 1.0 / (double)kSumScale;
    auto put = [&](int idx, int n0, int k0, auto w) { fill_tile(img, idx, n0, k0, w); };
    // local_0 with the embeddings folded in: columns [x_hi (Dc) | x_lo (Dc) | onehot (S)]
    auto w_local0 = [&](int o, int kc) -> double {
        const float* w0 = W + Lo.local0_w + (size_t)o * K0;
        if (kc < 2 * Dc) {
            const int j = kc % Dc;
            double acc = 0;
            for (int c = 0; c < C; ++c) acc += (double)w0[T + c] * W[Lo.emb_cont_w + (size_t)c * Dc + j];
            return acc;
        }
        const int s = kc - 2 * Dc;
        if (s >= S) return 0.0;
        double acc = 0;
        for (int dd = 0; dd < D; ++dd) acc += (double)w0[T + C + dd] * W[Lo.emb_disc + (size_t)s * D + dd];
        return acc;
    };
    for (int j = 0; j < 2; ++j) {
        put(LY::t_local0 + j, 8 * j, 0, w_local0);
        // projection globals: global_0 [H][mean H | sum H | T], global_1 [H][H], global_2 [G][H]
        put(LY::t_g0 + j, 8 * j, 0, [&](int o, int kc) { return (double)W[Lo.global0_w + (size_t)o * (2 * H + TX) + kc]; });
        put(LY::t_g0 + 2 + j, 8 * j, 0, [&](int o, int kc) { return inv_scale * W[Lo.global0_w + (size_t)o * (2 * H + TX) + H + kc]; });
        put(LY::t_g1 + j, 8 * j, 0, [&](int o, int kc) { return (double)W[Lo.global1_w + (size_t)o * H + kc]; });
    }
    for (int j = 0; j < 2 * GT; ++j)
        put(LY::t_g2 + j, 8 * j, 0, [&](int o, int kc) { return o < G ? (double)W[Lo.global2_w + (size_t)o * H + kc] : 0.0; });
    fill_vec(quads, LY::v_g1, [&](int i) { return W[Lo.global1_b + i]; });
    for (int gt = 0; gt < GT; ++gt) fill_vec(quads, LY::v_g2 + gt, [&](int i) { return 16 * gt + i < G ? W[Lo.global2_b + 16 * gt + i] : 0.0f; });
    for (int l = 0; l < L; ++l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        const int tl = LY::t_layer0 + l * LY::layer_tiles, vl = LY::v_layer0 + l * LY::layer_vecs;
        const int Kg = 2 * H + G + TX, Kl = H + G + TX;
        for (int j = 0; j < 2; ++j) {
            put(tl + LY::o_g1 + j, 8 * j, 0, [&](int o, int kc) { return (double)Wl[Lo.l_g1_w + (size_t)o * Kg + kc]; });
            put(tl + LY::o_g1 + 2 + j, 8 * j, 0, [&](int o, int kc) { return inv_scale * Wl[Lo.l_g1_w + (size_t)o * Kg + H + kc]; });
            for (int gt = 0; gt < GT; ++gt) {
                put(tl + LY::o_g1 + 4 + 2 * gt + j, 8 * j, 16 * gt,
                    [&](int o, int kc) { return kc < G ? (double)Wl[Lo.l_g1_w + (size_t)o * Kg + 2 * H + kc] : 0.0; });
                put(tl + LY::o_l1g + 2 * gt + j, 8 * j, 16 * gt,
                    [&](int o, int kc) { return kc < G ? (double)Wl[Lo.l_l1_w + (size_t)o * Kl + H + kc] : 0.0; });
            }
            put(tl + LY::o_l1 + j, 8 * j, 0, [&](int o, int kc) { return (double)Wl[Lo.l_l1_w + (size_t)o * Kl + kc]; });
            put(tl + LY::o_l2 + j, 8 * j, 0, [&](int o, int kc) { return (double)Wl[Lo.l_l2_w + (size_t)o * H + kc]; });
        }
        for (int j = 0; j < 2 * GT; ++j)
            put(tl + LY::o_g2 + j, 8 * j, 0, [&](int o, int kc) { return o < G ? (double)Wl[Lo.l_g2_w + (size_t)o * H + kc] : 0.0; });
        for (int gt = 0; gt < GT; ++gt)
            fill_vec(quads, vl + LY::ov_g2 + gt, [&](int i) { return 16 * gt + i < G ? Wl[Lo.l_g2_b + 16 * gt + i] : 0.0f; });
        fill_vec(quads, vl + LY::ov_l2, [&](int i) { return Wl[Lo.l_l2_b + i]; });
    }
    // output layer: n-tile 0 = head pre-activation F1 (W_out z-rows) (or the raw logits without a head), n-tile 1 = velocity rows
    const int tt = LY::t_layer0 + L * LY::layer_tiles, vt = LY::v_layer0 + L * LY::layer_vecs;
    std::vector<float> b_out(16, 0.0f), b_h2(16, 0.0f);
    if (Sh) {
        put(tt, 0, 0, [&](int j, int kc) {
            if (j >= Sh) return 0.0;
            double acc = 0;
            for (int s = 0; s < S; ++s) acc += (double)W[Lo.head0_w + (size_t)j * S + s] * W[Lo.out_w + (size_t)(Dc + s) * H + kc];
            return acc;
        });
        for (int j = 0; j < Sh; ++j) {
            double acc = W[Lo.head0_b + j];
            for (int s = 0; s < S; ++s) acc += (double)W[Lo.head0_w + (size_t)j * S + s] * W[Lo.out_b + Dc + s];
            b_out[j] = (float)acc;
        }
        put(tt + 2, 0, 0, [&](int o, int kc) { return (o < S && kc < Sh) ? (double)W[Lo.head2_w + (size_t)o * Sh + kc] : 0.0; });
        for (int o = 0; o < S; ++o) b_h2[o] = W[Lo.head2_b + o];
    } else {
        put(tt, 0, 0, [&](int o, int kc) { return o < S ? (double)W[Lo.out_w + (size_t)(Dc + o) * H + kc] : 0.0; });
        for (int o = 0; o < S; ++o) b_out[o] = W[Lo.out_b + Dc + o];
    }
    put(tt + 1, 0, 0, [&](int o, int kc) { return o < Dc ? (double)W[Lo.out_w + (size_t)o * H + kc] : 0.0; });
    for (int o = 0; o < Dc; ++o) b_out[8 + o] = W[Lo.out_b + o];
    fill_vec(quads, vt, [&](int i) { return b_out[i]; });
    fill_vec(quads, vt + 1, [&](int i) { return b_h2[i]; });

    const size_t nb = img.size() * sizeof(uint16_t), nf = quads.size() * sizeof(float);
    uint8_t* dev = nullptr;
    if (int rc = cuda_ok(cudaMalloc(&dev, nb + nf), "cudaMalloc mma image")) return rc;
    int rc = cuda_ok(cudaMemcpy(dev, img.data(), nb, cudaMemcpyHostToDevice), "mma image upload");
    if (!rc) rc = cuda_ok(cudaMemcpy(dev + nb, quads.data(), nf, cudaMemcpyHostToDevice), "mma image upload");
    if (rc) { cudaFree(dev); return rc; }
    *out = dev;
    *out_bytes = nb + nf;
    return MMB_OK;
}

template <int GT>
size_t smem_bytes(int L) {
    return ((Lay<GT>::image_bytes(L) + 127) & ~(size_t)127) + (size_t)kW * (kStageBytes + kSkipBytes) + (size_t)kW * kPoolFloats * 4;
}

template <int DC, int S, int SH, int GT>
int launch_kernel(const MmaParams& p, int grid, cudaStream_t stream) {
    const size_t bytes = smem_bytes<GT>(p.L);
    auto kern = p.x_in ? (p.cvec ? epic_mma_generate_kernel<DC, S, SH, GT, true, true> : epic_mma_generate_kernel<DC, S, SH, GT, true, false>)
                       : (p.cvec ? epic_mma_generate_kernel<DC, S, SH, GT, false, true> : epic_mma_generate_kernel<DC, S, SH, GT, false, false>);
    if (int rc = cuda_ok(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), "mma smem attribute")) return rc;
    kern<<<grid, kW * 32, bytes, stream>>>(p);
    return cuda_ok(cudaGetLastError(), "epic_mma launch");
}

int dispatch(const MmbEpicDims& d, const MmaParams& p, int grid, cudaStream_t stream) {
    const int sh = d.disc_head_hidden, gt = (d.dim_hidden_glob + 15) / 16;
    if (d.vocab_size == 8 && sh == 8 && gt == 1) return launch_kernel<3, 8, 8, 1>(p, grid, stream);
    if (d.vocab_size == 8 && sh == 0 && gt == 1) return launch_kernel<3, 8, 0, 1>(p, grid, stream);
    if (d.vocab_size == 8 && sh == 8 && gt == 2) return launch_kernel<3, 8, 8, 2>(p, grid, stream);
    if (d.vocab_size == 8 && sh == 0 && gt == 2) return launch_kernel<3, 8, 0, 2>(p, grid, stream);
    if (d.vocab_size == 4 && sh == 4 && gt == 1) return launch_kernel<3, 4, 4, 1>(p, grid, stream);
    if (d.vocab_size == 4 && sh == 0 && gt == 1) return launch_kernel<3, 4, 0, 1>(p, grid, stream);
    return fail(MMB_EUNSUPPORTED, "warp-MMA engine instantiated for Dc=3, (S, head) in {(8,8),(8,0),(4,4),(4,0)}, G<=16 (S=8: G<=32)");
}

}  // namespace

bool mma_supported(const MmbEpicDims* d, int N) {
    const bool head_ok = d->disc_head_hidden == 0 || d->disc_head_hidden == d->vocab_size;
    const int gt = (d->dim_hidden_glob + 15) / 16;
    return d->dim_hidden_local == kH && d->dim_hidden_glob >= 1 && gt <= (d->vocab_size == 8 ? 2 : 1) && d->dim_time_emb >= 1 &&
           d->num_blocks >= 1 && d->num_blocks <= kMaxL && d->dim_continuous == 3 && (d->vocab_size == 8 || d->vocab_size == 4) &&
           head_ok && N >= 1 && N <= kRowsPerWarp * kMaxCls && d->dim_context >= 0;
}

int mma_build_images(EpicModel* m, const float* packed_host) {
    const int gt = (m->dims.dim_hidden_glob + 15) / 16;
    return gt == 1 ? build_image_gt<1>(m->dims, m->layout, packed_host, &m->mma_image_f16, &m->mma_image_f16_bytes)
                   : build_image_gt<2>(m->dims, m->layout, packed_host, &m->mma_image_f16, &m->mma_image_f16_bytes);
}

// scratch (4-byte units): time-vector quads [n_steps][2 + 2L][8] float4 | context quads [B][1 + 2L][8] float4 (models with context
// features) | counts [16] | cursors [16] | jet_cnt [B] | lists [kKeys][B]
static size_t tvec_floats(const MmbEpicDims* d, int n_steps) { return (size_t)n_steps * (2 + 2 * d->num_blocks) * 32; }
static size_t cvec_floats(const MmbEpicDims* d, int B) { return d->dim_context > 0 ? (size_t)(B > 0 ? B : 0) * (1 + 2 * d->num_blocks) * 32 : 0; }
size_t mma_generate_scratch_floats(const MmbEpicDims* d, int n_steps, int B) {
    return tvec_floats(d, n_steps) + cvec_floats(d, B) + kCounterInts + (size_t)(B > 0 ? B : 0) * (1 + kKeys) + 16;
}

int launch_generate_mma(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* context, const float* dev_table, float* scratch,
                        int n_steps, float dt, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                        int B, int N, cudaStream_t stream, const MmaHostIO* host) {
    if (B == 0 || n_steps == 0) return MMB_OK;
    if (!m->mma_image_f16) return fail(MMB_EUNSUPPORTED, "warp-MMA engine: no operand image for this model");
    if ((reinterpret_cast<uintptr_t>(scratch) & 15) != 0) return fail(MMB_EINVAL, "mmb_generate: workspace must be 16-byte aligned");
    MmaParams p{};
    p.image = static_cast<const uint8_t*>(m->mma_image_f16);
    p.L = m->dims.num_blocks; p.skip = m->dims.skip_connection;
    p.x = x; p.k = k; p.mask = mask;
    if (host) {   // direct mode: sources from / results to mapped host memory
        p.x = host->x_out; p.k = nullptr; p.x_in = host->x_in; p.k_in = host->k_in; p.k_out = host->k_out; p.bad_tokens = host->bad_tokens;
    }
    p.step_tab = dev_table;
    p.n_steps = n_steps; p.dt = dt; p.u_jump = u_jump; p.seed = seed; p.jet_offset = jet_offset;
    p.B = B; p.N = N;
    if ((m->dims.dim_context > 0) != (context != nullptr))
        return fail(MMB_EINVAL, "mmb_generate: the model has %d context features, context pointer %s", m->dims.dim_context, context ? "given" : "missing");
    float4* cvec = context ? reinterpret_cast<float4*>(scratch + tvec_floats(&m->dims, n_steps)) : nullptr;
    int32_t* counts = reinterpret_cast<int32_t*>(scratch + tvec_floats(&m->dims, n_steps) + cvec_floats(&m->dims, B));
    int32_t* cursors = counts + kKeys;
    int32_t* jet_cnt = counts + kCounterInts;
    int32_t* lists = jet_cnt + B;
    if (int rc = cuda_ok(cudaMemsetAsync(counts, 0, kCounterInts * sizeof(int32_t), stream), "mma counters")) return rc;
    const int bin_blocks = (B + kPrologueThreads - 1) / kPrologueThreads;
    const int ctx_blocks = context ? (int)(((size_t)B * (1 + 2 * m->dims.num_blocks) * 8 + kPrologueThreads - 1) / kPrologueThreads) : 0;
    mma_prologue_kernel<<<n_steps + ctx_blocks + bin_blocks, kPrologueThreads, 0, stream>>>(m->w, m->layout, m->dims, dev_table + (size_t)n_steps * 4, n_steps,
                                                                                reinterpret_cast<float4*>(scratch), context, cvec, ctx_blocks, mask, B, N, counts, lists,
                                                                                jet_cnt, p.x, k, host ? host->k_out : nullptr);
    if (int rc = cuda_ok(cudaGetLastError(), "mma prologue launch")) return rc;
    p.tvec = reinterpret_cast<const float4*>(scratch); p.cvec = cvec; p.counts = counts; p.cursors = cursors; p.lists = lists; p.jet_cnt = jet_cnt;
    // Persistent grid: kMinBlocks CTAs per SM at most.  Any grid finishes any amount of work (warps claim jets until the
    // lists are empty), so the size only matters for speed: a small call takes about 1.25 warps per jet (the JetClass-like
    // mean is 1.14), which lets the kernels of neighbouring pipeline slices (mmb_generate_host) share the GPU side by side.
    const int want = (int)(((size_t)B * 5 + 4 * kW - 1) / (4 * kW));
    const int grid = want < m->sm_count * kMinBlocks ? (want > 0 ? want : 1) : m->sm_count * kMinBlocks;
    return dispatch(m->dims, p, grid, stream);
}

}  // namespace mmb
