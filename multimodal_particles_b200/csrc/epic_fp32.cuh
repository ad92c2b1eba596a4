// epic_fp32.cuh — the EPiC network's forward on CUDA cores in fp32, any widths: the parity anchor.  One implementation serves
// the forward and generation kernels (epic_fp32.cu) and the loss-gradient kernel (epic_grad.cu), so the heads the gradient
// kernel differentiates are exactly those of mmb_epic_forward(precision = fp32).
//
// One CTA of kFp32Threads threads owns one jet; thread `tid` owns particles tid, tid+128, ...  Every operation is the same
// IEEE fp32 operation, in the same order, as oracle/mmb_oracle.c (epic_forward_jet), so outputs are bit-identical to the CPU
// oracle — this is what lets the parity tests demand equality instead of a tolerance at any size.  The fast path is epic_tc.cu.
//
// Reference lines: mp/models/architectures/utils.py:112-172, epic.py:136-241,
// mp/models/generative/multimodal_bridge_matching.py:90-113,199-216.
#pragma once

#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

constexpr int kFp32Threads = 128;

struct Fp32Dims {
    int Dc, S, T, C, D, H, G, L, skip, Sh;
    int X;   // embedded context features behind the time embedding in the per-jet context vector (MmbEpicDims::dim_context)
    int HS;  // row stride of the per-particle hidden rows in shared memory (odd: conflict-free private rows)
    int RS;  // row stride of the scratch rows in shared memory: max(H, Sh, Dc+S, C), odd
    // [time embedding | context] width, and the in-widths of local_0, fc_global1 and fc_local1
    __host__ __device__ int TX() const { return T + X; }
    __host__ __device__ int K0() const { return T + C + D; }
    __host__ __device__ int Kg() const { return 2 * H + G + TX(); }
    __host__ __device__ int Kl() const { return H + G + TX(); }
};

__host__ __device__ inline int odd(int v) { return v | 1; }
__host__ __device__ inline int imax(int a, int b) { return a > b ? a : b; }

inline Fp32Dims make_dims(const MmbEpicDims& d) {
    Fp32Dims f{d.dim_continuous, d.vocab_size, d.dim_time_emb, d.dim_cont_emb, d.dim_disc_emb,
               d.dim_hidden_local, d.dim_hidden_glob, d.num_blocks, d.skip_connection, d.disc_head_hidden, d.dim_context, 0, 0};
    f.HS = odd(f.H);
    f.RS = odd(imax(imax(f.H, f.Sh), imax(f.Dc + f.S, f.C)));
    return f;
}

inline int check_dims(const MmbEpicDims& d) {
    if (d.dim_continuous < 1 || d.dim_continuous > 8 || d.vocab_size < 1 || d.vocab_size > 32)
        return fail(MMB_EINVAL, "need 1 <= Dc <= 8 and 1 <= S <= 32 (got Dc=%d S=%d)", d.dim_continuous, d.vocab_size);
    if (d.dim_hidden_local < 1 || d.dim_hidden_glob < 1 || d.dim_time_emb < 1 || d.num_blocks < 0 || d.dim_context < 0)
        return fail(MMB_EINVAL, "bad EPiC widths");
    return MMB_OK;
}

// Where one forward keeps its state.  The forward and generation kernels carve it from shared memory and update it in place.
struct Fp32Bufs {
    static constexpr bool kRecord = false;
    float *temb, *pj, *pool, *g0, *g1, *xg, *skipg, *sum, *red, *xl, *skipl, *row;
    int* cnt;
};

// The loss-gradient kernel's state, in its CTA's region of global memory with dense rows of H.  Its forward also keeps every
// activation the backward reads: xl is [L+1][N][H] (layer l reads slice l and writes slice l+1, so the trunk skip is slice 0
// and skipl == xl), the per-layer fields are [L][...], the rest per particle or per jet.  Masked particles are skipped.
struct Fp32Record : Fp32Bufs {
    static constexpr bool kRecord = true;
    float *feat;                            // [N][K0] local_0's input row: [time embedding | continuous emb | discrete emb]
    float *a0;                              // [N][H] local_0's pre-activation
    float *g0p, *g1p, *xgp;                 // global_0..2 pre-activations
    float *lpool, *wp, *up, *lj, *p, *q;    // per layer: fc_global1's input, fc_global1 / fc_global2 pre-activations,
                                            // fc_local1's per-jet input [xg' | context], fc_local1 / fc_local2 + residual
    float *ho, *z, *r;                      // [N][Dc+S] output layer, [N][Sh] disc-head pre-activation and activation
};

// acc + sum_i w[i]*in[i], ascending i, one fmaf per term
__device__ __forceinline__ float dot_from(float acc, const float* __restrict__ w, const float* in, int n) {
    for (int i = 0; i < n; ++i) acc = __fmaf_rn(__ldg(w + i), in[i], acc);
    return acc;
}

// four output rows at once (same chains, inputs read once)
__device__ __forceinline__ void dot4_from(float (&acc)[4], const float* __restrict__ w, int ldw, const float* in, int n) {
    const float *w0 = w, *w1 = w + ldw, *w2 = w + 2 * ldw, *w3 = w + 3 * ldw;
    for (int i = 0; i < n; ++i) {
        const float a = in[i];
        acc[0] = __fmaf_rn(__ldg(w0 + i), a, acc[0]);
        acc[1] = __fmaf_rn(__ldg(w1 + i), a, acc[1]);
        acc[2] = __fmaf_rn(__ldg(w2 + i), a, acc[2]);
        acc[3] = __fmaf_rn(__ldg(w3 + i), a, acc[3]);
    }
}

// masked sum over particles of column o of rows [N][ld] for all o < H, in the oracle's tree order (tree_sum()):
// lane partial (ascending n, from +0) -> xor butterfly per warp -> warps in order.
__device__ inline void pooled_sums(const float* rows, int ld, const uint8_t* mask, int N, int H, float* red, float* sum) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int o = 0; o < H; ++o) {
        float part = 0.0f;
        for (int n = tid; n < N; n += kFp32Threads)
            part = __fadd_rn(part, __fmul_rn(rows[(size_t)n * ld + o], (float)mask[n]));
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if (lane == 0) red[warp * H + o] = part;
    }
    __syncthreads();
    for (int o = tid; o < H; o += kFp32Threads)
        sum[o] = __fadd_rn(__fadd_rn(__fadd_rn(red[o], red[H + o]), red[2 * H + o]), red[3 * H + o]);
    __syncthreads();
}

// One network evaluation for the jet held by this CTA; s.temb holds the jet's [time embedding | context] on entry.  x/k/mask
// point to the jet's current state (global or shared).  Heads go to v_out/logits_out/hidden_out (global or shared; hidden
// nullable); with Bufs = Fp32Record the output layer goes to s.ho instead of v_out, and masked particles are skipped.  Live
// particles see the same operations either way.
template <class Bufs>
__device__ void epic_forward_jet(const float* __restrict__ W, const MmbEpicLayout& Lo, const Fp32Dims& f, const Bufs& s,
                                 const float* x, const uint8_t* k, const uint8_t* mask, int N,
                                 float* v_out, float* logits_out, float* hidden_out) {
    constexpr bool kRecord = Bufs::kRecord;
    const int tid = threadIdx.x;
    const int Dc = f.Dc, S = f.S, T = f.T, C = f.C, D = f.D, H = f.H, G = f.G, Sh = f.Sh;
    const int K0 = f.K0();
    const int TX = f.TX();   // only the time part of s.temb is among the particle features (utils.py:139-145)
    const int HS = kRecord ? H : f.HS, RS = kRecord ? H : f.RS;   // hidden / scratch row strides

    // per-jet part of local_0, particle count
    for (int o = tid; o < H; o += kFp32Threads)
        s.pj[o] = dot_from(__ldg(W + Lo.local0_b + o), W + Lo.local0_w + (size_t)o * K0, s.temb, T);
    {
        int c = 0;
        for (int n = tid; n < N; n += kFp32Threads) c += mask[n] ? 1 : 0;
        c = __reduce_add_sync(0xffffffffu, c);
        if ((tid & 31) == 0) s.cnt[tid >> 5] = c;
    }
    __syncthreads();
    const float cnt = (float)(s.cnt[0] + s.cnt[1] + s.cnt[2] + s.cnt[3]);

    // ---- InputEmbeddings + local_0 (utils.py:133-172, epic.py:186); xl holds lrelu(.) UNmasked here
    for (int n = tid; n < N; n += kFp32Threads) {
        float* xn = s.xl + (size_t)n * HS;
        if (mask[n]) {
            float* emb = s.row + (size_t)n * RS;
            if constexpr (kRecord) emb = s.feat + (size_t)n * K0 + T;
            for (int c = 0; c < C; ++c)
                emb[c] = dot_from(__ldg(W + Lo.emb_cont_b + c), W + Lo.emb_cont_w + (size_t)c * Dc, x + (size_t)n * Dc, Dc);
            const float* e = W + Lo.emb_disc + (size_t)k[n] * D;
            if constexpr (kRecord) {
                for (int t = 0; t < T; ++t) s.feat[(size_t)n * K0 + t] = s.temb[t];
                for (int d = 0; d < D; ++d) emb[C + d] = __ldg(e + d);
            }
            for (int o = 0; o < H; ++o) {
                const float* w = W + Lo.local0_w + (size_t)o * K0;
                float acc = dot_from(s.pj[o], w + T, emb, C);
                for (int d = 0; d < D; ++d) acc = __fmaf_rn(__ldg(w + T + C + d), __ldg(e + d), acc);
                if constexpr (kRecord) s.a0[(size_t)n * H + o] = acc;
                xn[o] = lrelu(acc);
            }
        } else {
            for (int o = 0; o < H; ++o) xn[o] = lrelu(__ldg(W + Lo.local0_b + o));
        }
    }
    __syncthreads();
    // ---- meansum_pool + global_0..2 (epic.py:136-143,187-190)
    pooled_sums(s.xl, HS, mask, N, H, s.red, s.sum);
    for (int o = tid; o < H; o += kFp32Threads) {
        s.pool[o] = __fdiv_rn(s.sum[o], cnt);
        s.pool[H + o] = s.sum[o];
    }
    for (int i = tid; i < TX; i += kFp32Threads) s.pool[2 * H + i] = s.temb[i];
    __syncthreads();
    for (int o = tid; o < H; o += kFp32Threads) {
        const float a = dot_from(__ldg(W + Lo.global0_b + o), W + Lo.global0_w + (size_t)o * (2 * H + TX), s.pool, 2 * H + TX);
        if constexpr (kRecord) s.g0p[o] = a;
        s.g0[o] = lrelu(a);
    }
    __syncthreads();
    for (int o = tid; o < H; o += kFp32Threads) {
        const float a = dot_from(__ldg(W + Lo.global1_b + o), W + Lo.global1_w + (size_t)o * H, s.g0, H);
        if constexpr (kRecord) s.g1p[o] = a;
        s.g1[o] = lrelu(a);
    }
    __syncthreads();
    for (int o = tid; o < G; o += kFp32Threads) {
        const float a = dot_from(__ldg(W + Lo.global2_b + o), W + Lo.global2_w + (size_t)o * H, s.g1, H);
        if constexpr (kRecord) s.xgp[o] = a;
        s.xg[o] = lrelu(a);
        if (f.skip) s.skipg[o] = s.xg[o];
    }
    // x_local * mask, skip copies (epic.py:148-149,191)
    for (int n = tid; n < N; n += kFp32Threads) {
        const float m = (float)mask[n];
        float* xn = s.xl + (size_t)n * HS;
        for (int o = 0; o < H; ++o) {
            xn[o] = __fmul_rn(xn[o], m);
            if (!kRecord && f.skip) s.skipl[(size_t)n * HS + o] = xn[o];
        }
    }
    __syncthreads();

    // ---- EPiC layers (epic.py:217-241,152-155)
    for (int l = 0; l < f.L; ++l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        float *xin = s.xl, *xout = s.xl, *pool = s.pool, *xgn = s.g0;
        float *wp = nullptr, *up = nullptr, *p = nullptr, *q = nullptr;
        const int Kg = f.Kg(), Kl = f.Kl();
        if constexpr (kRecord) {
            xin = s.xl + (size_t)l * N * H;
            xout = xin + (size_t)N * H;
            pool = s.lpool + (size_t)l * Kg;
            xgn = s.lj + (size_t)l * (G + TX);
            wp = s.wp + (size_t)l * H;
            up = s.up + (size_t)l * G;
            p = s.p + (size_t)l * N * H;
            q = s.q + (size_t)l * N * H;
        }
        pooled_sums(xin, HS, mask, N, H, s.red, s.sum);
        for (int o = tid; o < H; o += kFp32Threads) {
            pool[o] = __fdiv_rn(s.sum[o], cnt);
            pool[H + o] = s.sum[o];
        }
        for (int i = tid; i < G; i += kFp32Threads) pool[2 * H + i] = s.xg[i];
        for (int i = tid; i < TX; i += kFp32Threads) pool[2 * H + G + i] = s.temb[i];
        __syncthreads();
        for (int o = tid; o < H; o += kFp32Threads) {
            const float a = dot_from(__ldg(Wl + Lo.l_g1_b + o), Wl + Lo.l_g1_w + (size_t)o * Kg, pool, Kg);
            if constexpr (kRecord) wp[o] = a;
            s.g1[o] = lrelu(a);
        }
        __syncthreads();
        for (int o = tid; o < G; o += kFp32Threads) {
            const float a = __fadd_rn(dot_from(__ldg(Wl + Lo.l_g2_b + o), Wl + Lo.l_g2_w + (size_t)o * H, s.g1, H), s.xg[o]);
            if constexpr (kRecord) up[o] = a;
            xgn[o] = lrelu(a);
        }
        if constexpr (kRecord)
            for (int i = tid; i < TX; i += kFp32Threads) xgn[G + i] = s.temb[i];
        __syncthreads();
        for (int o = tid; o < G; o += kFp32Threads) s.xg[o] = xgn[o];
        __syncthreads();
        for (int o = tid; o < H; o += kFp32Threads) {
            const float* w = Wl + Lo.l_l1_w + (size_t)o * Kl;
            float acc = dot_from(__ldg(Wl + Lo.l_l1_b + o), w + H, s.xg, G);
            s.pj[o] = dot_from(acc, w + H + G, s.temb, TX);
        }
        __syncthreads();
        for (int n = tid; n < N; n += kFp32Threads) {
            if constexpr (kRecord)
                if (!mask[n]) {   // a masked particle's row only ever enters a sum multiplied by its zero mask
                    for (int o = 0; o < H; ++o) xout[(size_t)n * H + o] = 0.0f;
                    continue;
                }
            const float m = (float)mask[n];
            const float* xn = xin + (size_t)n * HS;
            float* xo = xout + (size_t)n * HS;
            float* l1 = s.row + (size_t)n * RS;
            int o = 0;
            for (; o + 4 <= H; o += 4) {
                float acc[4] = {s.pj[o], s.pj[o + 1], s.pj[o + 2], s.pj[o + 3]};
                dot4_from(acc, Wl + Lo.l_l1_w + (size_t)o * Kl, Kl, xn, H);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if constexpr (kRecord) p[(size_t)n * H + o + j] = acc[j];
                    l1[o + j] = lrelu(acc[j]);
                }
            }
            for (; o < H; ++o) {
                const float a = dot_from(s.pj[o], Wl + Lo.l_l1_w + (size_t)o * Kl, xn, H);
                if constexpr (kRecord) p[(size_t)n * H + o] = a;
                l1[o] = lrelu(a);
            }
            // fc_local2 + residual, mask, trunk skip.  In place, new values overwrite xn only after all H are known.
            for (o = 0; o + 4 <= H; o += 4) {
                float acc[4] = {__ldg(Wl + Lo.l_l2_b + o), __ldg(Wl + Lo.l_l2_b + o + 1), __ldg(Wl + Lo.l_l2_b + o + 2),
                                __ldg(Wl + Lo.l_l2_b + o + 3)};
                dot4_from(acc, Wl + Lo.l_l2_w + (size_t)o * H, H, l1, H);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float a = __fadd_rn(acc[j], xn[o + j]);
                    if constexpr (kRecord) q[(size_t)n * H + o + j] = a;
                    float val = __fmul_rn(lrelu(a), m);
                    if (f.skip) val = __fadd_rn(val, s.skipl[(size_t)n * HS + o + j]);
                    xo[o + j] = val;  // safe in place: fc_local2 reads l1, the residual reads xn[o+j] only
                }
            }
            for (; o < H; ++o) {
                const float a = __fadd_rn(dot_from(__ldg(Wl + Lo.l_l2_b + o), Wl + Lo.l_l2_w + (size_t)o * H, l1, H), xn[o]);
                if constexpr (kRecord) q[(size_t)n * H + o] = a;
                float val = __fmul_rn(lrelu(a), m);
                if (f.skip) val = __fadd_rn(val, s.skipl[(size_t)n * HS + o]);
                xo[o] = val;
            }
        }
        if (f.skip)
            for (int o = tid; o < G; o += kFp32Threads) s.xg[o] = __fadd_rn(s.xg[o], s.skipg[o]);
        __syncthreads();
    }

    // ---- output layer + heads (epic.py:158-162, mbm.py:105-113)
    const float* xlast = kRecord ? s.xl + (size_t)f.L * N * H : s.xl;
    for (int n = tid; n < N; n += kFp32Threads) {
        if constexpr (kRecord)
            if (!mask[n]) continue;
        const float m = (float)mask[n];
        const float* xn = xlast + (size_t)n * HS;
        float* r = s.row + (size_t)n * RS;  // z1[Sh]
        float hl[40];
        float* h = hl;
        if constexpr (kRecord) {
            r = s.r + (size_t)n * Sh;
            h = s.ho + (size_t)n * (Dc + S);
        }
        for (int o = 0; o < Dc + S; ++o)
            h[o] = __fmul_rn(dot_from(__ldg(W + Lo.out_b + o), W + Lo.out_w + (size_t)o * H, xn, H), m);
        if constexpr (!kRecord)
            for (int c = 0; c < Dc; ++c) v_out[(size_t)n * Dc + c] = h[c];
        if (Sh) {
            for (int o = 0; o < Sh; ++o) {
                const float a = dot_from(__ldg(W + Lo.head0_b + o), W + Lo.head0_w + (size_t)o * S, h + Dc, S);
                if constexpr (kRecord) s.z[(size_t)n * Sh + o] = a;
                r[o] = selu(a);
            }
            for (int o = 0; o < S; ++o)
                logits_out[(size_t)n * S + o] = dot_from(__ldg(W + Lo.head2_b + o), W + Lo.head2_w + (size_t)o * Sh, r, Sh);
        } else {
            for (int o = 0; o < S; ++o) logits_out[(size_t)n * S + o] = h[Dc + o];
        }
        if (hidden_out)
            for (int o = 0; o < H; ++o) hidden_out[(size_t)n * H + o] = xn[o];
    }
}

}  // namespace mmb
