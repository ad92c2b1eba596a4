// epic_fp32.cu — EPiC network on CUDA cores in fp32, any widths; the parity anchor.
//
// One CTA of 128 threads owns one jet; thread `tid` owns particles tid, tid+128, ...  Every
// operation is the same IEEE fp32 operation, in the same order, as oracle/mmb_oracle.c
// (epic_forward_jet), so outputs are bit-identical to the CPU oracle — this is what lets the
// parity tests demand equality instead of a tolerance at any size.  The fast path is epic_tc.cu.
//
// Reference lines: mp/models/architectures/utils.py:112-172, epic.py:136-241,
// mp/models/generative/multimodal_bridge_matching.py:90-113,199-216.
#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

namespace {

constexpr int kThreads = 128;

struct Fp32Dims {
    int Dc, S, T, C, D, H, G, L, skip, Sh;
    int X;   // embedded context features behind the time embedding in the per-jet context vector (MmbEpicDims::dim_context)
    int HS;  // row stride of the per-particle hidden rows (odd: conflict-free private rows)
    int RS;  // row stride of the scratch rows: max(H, Sh, Dc+S, C), odd
};

__host__ __device__ inline int odd(int v) { return v | 1; }
__host__ __device__ inline int imax(int a, int b) { return a > b ? a : b; }

__host__ Fp32Dims make_dims(const MmbEpicDims& d) {
    Fp32Dims f{d.dim_continuous, d.vocab_size, d.dim_time_emb, d.dim_cont_emb, d.dim_disc_emb,
               d.dim_hidden_local, d.dim_hidden_glob, d.num_blocks, d.skip_connection, d.disc_head_hidden, d.dim_context, 0, 0};
    f.HS = odd(f.H);
    f.RS = odd(imax(imax(f.H, f.Sh), imax(f.Dc + f.S, f.C)));
    return f;
}

// shared-memory carve-up (floats)
struct Smem {
    float *temb, *pj, *pool, *g0, *g1, *xg, *skipg, *sum, *red, *xl, *skipl, *row;
    int* cnt;
};

__host__ __device__ inline size_t smem_floats(const Fp32Dims& f, int N) {
    return (size_t)(f.T + f.X) + f.H + (2 * f.H + f.G + f.T + f.X) + f.H + f.H + f.G + f.G + f.H + 4 * f.H + 8 +
           (size_t)N * f.HS * 2 + (size_t)N * f.RS;
}

__device__ inline Smem carve(float* base, const Fp32Dims& f, int N) {
    Smem s;
    float* p = base;
    s.temb = p; p += f.T + f.X;   // [time embedding | embedded context]: the reference's `context` vector (utils.py:166-170)
    s.pj = p; p += f.H;
    s.pool = p; p += 2 * f.H + f.G + f.T + f.X;
    s.g0 = p; p += f.H;
    s.g1 = p; p += f.H;
    s.xg = p; p += f.G;
    s.skipg = p; p += f.G;
    s.sum = p; p += f.H;
    s.red = p; p += 4 * f.H;
    s.cnt = reinterpret_cast<int*>(p); p += 8;
    s.xl = p; p += (size_t)N * f.HS;
    s.skipl = p; p += (size_t)N * f.HS;
    s.row = p;
    return s;
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

// masked sum over particles of column o for all o < H, in the oracle's tree order (tree_sum()):
// lane partial (ascending n, from +0) -> xor butterfly per warp -> warps in order.
__device__ void pooled_sums(const Smem& s, const Fp32Dims& f, const uint8_t* mask, int N) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int o = 0; o < f.H; ++o) {
        float part = 0.0f;
        for (int n = tid; n < N; n += kThreads)
            part = __fadd_rn(part, __fmul_rn(s.xl[(size_t)n * f.HS + o], (float)mask[n]));
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if (lane == 0) s.red[warp * f.H + o] = part;
    }
    __syncthreads();
    for (int o = tid; o < f.H; o += kThreads)
        s.sum[o] = __fadd_rn(__fadd_rn(__fadd_rn(s.red[o], s.red[f.H + o]), s.red[2 * f.H + o]), s.red[3 * f.H + o]);
    __syncthreads();
}

// One network evaluation for the jet held by this CTA.  x/k/mask point to the jet's current state
// (global or shared).  Outputs go to v_out/logits_out/hidden_out (global or shared; hidden nullable).
__device__ void epic_forward_jet(const float* __restrict__ W, const MmbEpicLayout& Lo, const Fp32Dims& f, const Smem& s,
                                 const float* x, const uint8_t* k, const uint8_t* mask, int N,
                                 float* v_out, float* logits_out, float* hidden_out) {
    const int tid = threadIdx.x;
    const int Dc = f.Dc, S = f.S, T = f.T, C = f.C, D = f.D, H = f.H, G = f.G, Sh = f.Sh;
    const int K0 = T + C + D;
    const int TX = T + f.X;   // only the time part of s.temb is among the particle features (utils.py:139-145)

    // per-jet part of local_0, particle count
    for (int o = tid; o < H; o += kThreads)
        s.pj[o] = dot_from(__ldg(W + Lo.local0_b + o), W + Lo.local0_w + (size_t)o * K0, s.temb, T);
    {
        int c = 0;
        for (int n = tid; n < N; n += kThreads) c += mask[n] ? 1 : 0;
        c = __reduce_add_sync(0xffffffffu, c);
        if ((tid & 31) == 0) s.cnt[tid >> 5] = c;
    }
    __syncthreads();
    const float cnt = (float)(s.cnt[0] + s.cnt[1] + s.cnt[2] + s.cnt[3]);

    // ---- InputEmbeddings + local_0 (utils.py:133-172, epic.py:186); xl holds lrelu(.) UNmasked here
    for (int n = tid; n < N; n += kThreads) {
        float* xn = s.xl + (size_t)n * f.HS;
        if (mask[n]) {
            float* emb = s.row + (size_t)n * f.RS;
            for (int c = 0; c < C; ++c)
                emb[c] = dot_from(__ldg(W + Lo.emb_cont_b + c), W + Lo.emb_cont_w + (size_t)c * Dc, x + (size_t)n * Dc, Dc);
            const float* e = W + Lo.emb_disc + (size_t)k[n] * D;
            for (int o = 0; o < H; ++o) {
                const float* w = W + Lo.local0_w + (size_t)o * K0;
                float acc = dot_from(s.pj[o], w + T, emb, C);
                for (int d = 0; d < D; ++d) acc = __fmaf_rn(__ldg(w + T + C + d), __ldg(e + d), acc);
                xn[o] = lrelu(acc);
            }
        } else {
            for (int o = 0; o < H; ++o) xn[o] = lrelu(__ldg(W + Lo.local0_b + o));
        }
    }
    __syncthreads();
    // ---- meansum_pool + global_0..2 (epic.py:136-143,187-190)
    pooled_sums(s, f, mask, N);
    for (int o = tid; o < H; o += kThreads) {
        s.pool[o] = __fdiv_rn(s.sum[o], cnt);
        s.pool[H + o] = s.sum[o];
    }
    for (int i = tid; i < TX; i += kThreads) s.pool[2 * H + i] = s.temb[i];
    __syncthreads();
    for (int o = tid; o < H; o += kThreads)
        s.g0[o] = lrelu(dot_from(__ldg(W + Lo.global0_b + o), W + Lo.global0_w + (size_t)o * (2 * H + TX), s.pool, 2 * H + TX));
    __syncthreads();
    for (int o = tid; o < H; o += kThreads)
        s.g1[o] = lrelu(dot_from(__ldg(W + Lo.global1_b + o), W + Lo.global1_w + (size_t)o * H, s.g0, H));
    __syncthreads();
    for (int o = tid; o < G; o += kThreads) {
        s.xg[o] = lrelu(dot_from(__ldg(W + Lo.global2_b + o), W + Lo.global2_w + (size_t)o * H, s.g1, H));
        if (f.skip) s.skipg[o] = s.xg[o];
    }
    // x_local * mask, skip copies (epic.py:148-149,191)
    for (int n = tid; n < N; n += kThreads) {
        const float m = (float)mask[n];
        float* xn = s.xl + (size_t)n * f.HS;
        for (int o = 0; o < H; ++o) {
            xn[o] = __fmul_rn(xn[o], m);
            if (f.skip) s.skipl[(size_t)n * f.HS + o] = xn[o];
        }
    }
    __syncthreads();

    // ---- EPiC layers (epic.py:217-241,152-155)
    for (int l = 0; l < f.L; ++l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        pooled_sums(s, f, mask, N);
        for (int o = tid; o < H; o += kThreads) {
            s.pool[o] = __fdiv_rn(s.sum[o], cnt);
            s.pool[H + o] = s.sum[o];
        }
        for (int i = tid; i < G; i += kThreads) s.pool[2 * H + i] = s.xg[i];
        for (int i = tid; i < TX; i += kThreads) s.pool[2 * H + G + i] = s.temb[i];
        __syncthreads();
        const int Kg = 2 * H + G + TX;
        for (int o = tid; o < H; o += kThreads)
            s.g1[o] = lrelu(dot_from(__ldg(Wl + Lo.l_g1_b + o), Wl + Lo.l_g1_w + (size_t)o * Kg, s.pool, Kg));
        __syncthreads();
        for (int o = tid; o < G; o += kThreads)
            s.g0[o] = lrelu(__fadd_rn(dot_from(__ldg(Wl + Lo.l_g2_b + o), Wl + Lo.l_g2_w + (size_t)o * H, s.g1, H), s.xg[o]));
        __syncthreads();
        for (int o = tid; o < G; o += kThreads) s.xg[o] = s.g0[o];
        __syncthreads();
        const int Kl = H + G + TX;
        for (int o = tid; o < H; o += kThreads) {
            const float* w = Wl + Lo.l_l1_w + (size_t)o * Kl;
            float acc = dot_from(__ldg(Wl + Lo.l_l1_b + o), w + H, s.xg, G);
            s.pj[o] = dot_from(acc, w + H + G, s.temb, TX);
        }
        __syncthreads();
        for (int n = tid; n < N; n += kThreads) {
            const float m = (float)mask[n];
            float* xn = s.xl + (size_t)n * f.HS;
            float* l1 = s.row + (size_t)n * f.RS;
            int o = 0;
            for (; o + 4 <= H; o += 4) {
                float acc[4] = {s.pj[o], s.pj[o + 1], s.pj[o + 2], s.pj[o + 3]};
                dot4_from(acc, Wl + Lo.l_l1_w + (size_t)o * Kl, Kl, xn, H);
#pragma unroll
                for (int j = 0; j < 4; ++j) l1[o + j] = lrelu(acc[j]);
            }
            for (; o < H; ++o) l1[o] = lrelu(dot_from(s.pj[o], Wl + Lo.l_l1_w + (size_t)o * Kl, xn, H));
            // fc_local2 + residual, mask, trunk skip.  New values overwrite xn only after all H are known.
            for (o = 0; o + 4 <= H; o += 4) {
                float acc[4] = {__ldg(Wl + Lo.l_l2_b + o), __ldg(Wl + Lo.l_l2_b + o + 1), __ldg(Wl + Lo.l_l2_b + o + 2),
                                __ldg(Wl + Lo.l_l2_b + o + 3)};
                dot4_from(acc, Wl + Lo.l_l2_w + (size_t)o * H, H, l1, H);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float val = __fmul_rn(lrelu(__fadd_rn(acc[j], xn[o + j])), m);
                    if (f.skip) val = __fadd_rn(val, s.skipl[(size_t)n * f.HS + o + j]);
                    xn[o + j] = val;  // safe: fc_local2 reads l1, the residual reads xn[o+j] only
                }
            }
            for (; o < H; ++o) {
                float val = dot_from(__ldg(Wl + Lo.l_l2_b + o), Wl + Lo.l_l2_w + (size_t)o * H, l1, H);
                val = __fmul_rn(lrelu(__fadd_rn(val, xn[o])), m);
                if (f.skip) val = __fadd_rn(val, s.skipl[(size_t)n * f.HS + o]);
                xn[o] = val;
            }
        }
        if (f.skip)
            for (int o = tid; o < G; o += kThreads) s.xg[o] = __fadd_rn(s.xg[o], s.skipg[o]);
        __syncthreads();
    }

    // ---- output layer + heads (epic.py:158-162, mbm.py:105-113)
    for (int n = tid; n < N; n += kThreads) {
        const float m = (float)mask[n];
        const float* xn = s.xl + (size_t)n * f.HS;
        float* r = s.row + (size_t)n * f.RS;  // h[Dc+S] then reused for z1[Sh]
        float h[40];
        for (int o = 0; o < Dc + S; ++o)
            h[o] = __fmul_rn(dot_from(__ldg(W + Lo.out_b + o), W + Lo.out_w + (size_t)o * H, xn, H), m);
        for (int c = 0; c < Dc; ++c) v_out[(size_t)n * Dc + c] = h[c];
        if (Sh) {
            for (int o = 0; o < Sh; ++o)
                r[o] = selu(dot_from(__ldg(W + Lo.head0_b + o), W + Lo.head0_w + (size_t)o * S, h + Dc, S));
            for (int o = 0; o < S; ++o)
                logits_out[(size_t)n * S + o] = dot_from(__ldg(W + Lo.head2_b + o), W + Lo.head2_w + (size_t)o * Sh, r, Sh);
        } else {
            for (int o = 0; o < S; ++o) logits_out[(size_t)n * S + o] = h[Dc + o];
        }
        if (hidden_out)
            for (int o = 0; o < H; ++o) hidden_out[(size_t)n * H + o] = xn[o];
    }
}

__global__ void __launch_bounds__(kThreads)
epic_forward_fp32_kernel(const float* __restrict__ W, MmbEpicLayout Lo, Fp32Dims f,
                         const float* __restrict__ x, const uint8_t* __restrict__ k, const uint8_t* __restrict__ mask,
                         const float* __restrict__ temb, int temb_stride, int N,
                         float* __restrict__ v_out, float* __restrict__ logits_out, float* __restrict__ hidden_out) {
    extern __shared__ float smem[];
    const Smem s = carve(smem, f, N);
    const size_t b = blockIdx.x;
    for (int i = threadIdx.x; i < f.T + f.X; i += kThreads) s.temb[i] = temb[b * temb_stride + i];
    __syncthreads();
    epic_forward_jet(W, Lo, f, s, x + b * N * f.Dc, k + b * N, mask + b * N, N,
                     v_out + b * N * f.Dc, logits_out + b * N * f.S, hidden_out ? hidden_out + b * N * f.H : nullptr);
}

// Whole generation for one jet per CTA, state in shared memory across all steps
// (MultiModalBridgeMatching.simulate_dynamics, mbm.py:199-216).
__global__ void __launch_bounds__(kThreads)
generate_fp32_kernel(const float* __restrict__ W, MmbEpicLayout Lo, Fp32Dims f,
                     float* __restrict__ x, uint8_t* __restrict__ k, const uint8_t* __restrict__ mask,
                     const float* __restrict__ context, const float* __restrict__ table, int n_steps, float dt,
                     const float* __restrict__ u_jump, uint64_t seed, uint64_t jet_offset, int B, int N) {
    extern __shared__ float smem[];
    const Smem s = carve(smem, f, N);
    float* sx = smem + smem_floats(f, N);
    float* sv = sx + (size_t)N * f.Dc;
    float* slog = sv + (size_t)N * f.Dc;
    uint8_t* sk = reinterpret_cast<uint8_t*>(slog + (size_t)N * f.S);
    uint8_t* sm = sk + ((N + 15) & ~15);
    const size_t b = blockIdx.x;
    const int tid = threadIdx.x;
    for (int i = tid; i < N * f.Dc; i += kThreads) sx[i] = x[b * N * f.Dc + i];
    for (int n = tid; n < N; n += kThreads) { sk[n] = k[b * N + n]; sm[n] = mask[b * N + n]; }
    const float* temb_tab = table + (size_t)n_steps * 4;
    for (int i = tid; i < f.X; i += kThreads) s.temb[f.T + i] = context[b * f.X + i];   // constant over the steps (mbm.py:143-144)
    for (int step = 0; step < n_steps; ++step) {
        for (int i = tid; i < f.T; i += kThreads) s.temb[i] = temb_tab[(size_t)step * f.T + i];
        __syncthreads();
        epic_forward_jet(W, Lo, f, s, sx, sk, sm, N, sv, slog, nullptr);
        const StepScalars sc{dt, table[step * 4 + 0], table[step * 4 + 1], table[step * 4 + 2]};
        for (int n = tid; n < N; n += kThreads) {   // each particle is read and written by its owner only
            const int m = sm[n];
            for (int c = 0; c < f.Dc; ++c) sx[n * f.Dc + c] = euler(sx[n * f.Dc + c], sv[n * f.Dc + c], dt, (float)m);
            const float u = u_jump ? u_jump[((size_t)step * B + b) * N + n]
                                   : philox_uniform(seed, jet_offset + b, 0, step, n);
            sk[n] = (uint8_t)(telegraph_jump_rt(slog + (size_t)n * f.S, f.S, sk[n], u, sc) * m);
        }
        __syncthreads();
    }
    for (int i = tid; i < N * f.Dc; i += kThreads) x[b * N * f.Dc + i] = sx[i];
    for (int n = tid; n < N; n += kThreads) k[b * N + n] = sk[n];
}

int check_dims(const MmbEpicDims& d) {
    if (d.dim_continuous < 1 || d.dim_continuous > 8 || d.vocab_size < 1 || d.vocab_size > 32)
        return fail(MMB_EINVAL, "need 1 <= Dc <= 8 and 1 <= S <= 32 (got Dc=%d S=%d)", d.dim_continuous, d.vocab_size);
    if (d.dim_hidden_local < 1 || d.dim_hidden_glob < 1 || d.dim_time_emb < 1 || d.num_blocks < 0 || d.dim_context < 0)
        return fail(MMB_EINVAL, "bad EPiC widths");
    return MMB_OK;
}

}  // namespace

int launch_epic_forward_fp32(const EpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask,
                             const float* temb, int temb_stride, int B, int N,
                             float* v_out, float* logits_out, float* hidden_out, cudaStream_t stream) {
    if (int rc = check_dims(m->dims)) return rc;
    if (B == 0 || N == 0) return MMB_OK;
    const Fp32Dims f = make_dims(m->dims);
    const size_t bytes = smem_floats(f, N) * sizeof(float);
    if (bytes > 227 * 1024) return fail(MMB_ENOMEM, "fp32 EPiC kernel needs %zu B of shared memory (N=%d, H=%d)", bytes, N, f.H);
    if (int rc = cuda_ok(cudaFuncSetAttribute(epic_forward_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes),
                         "smem attribute"))
        return rc;
    epic_forward_fp32_kernel<<<B, kThreads, bytes, stream>>>(m->w, m->layout, f, x, k, mask, temb, temb_stride, N,
                                                               v_out, logits_out, hidden_out);
    return cuda_ok(cudaGetLastError(), "epic_forward_fp32 launch");
}

int launch_generate_fp32(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* context, const float* dev_table,
                         int n_steps, float dt, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                         int B, int N, cudaStream_t stream) {
    if (int rc = check_dims(m->dims)) return rc;
    if (B == 0 || N == 0 || n_steps == 0) return MMB_OK;
    const Fp32Dims f = make_dims(m->dims);
    const size_t bytes = (smem_floats(f, N) + (size_t)N * (2 * f.Dc + f.S)) * sizeof(float) + 2 * ((N + 15) & ~15);
    if (bytes > 227 * 1024) return fail(MMB_ENOMEM, "fp32 generate kernel needs %zu B of shared memory", bytes);
    if (int rc = cuda_ok(cudaFuncSetAttribute(generate_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes),
                         "smem attribute"))
        return rc;
    generate_fp32_kernel<<<B, kThreads, bytes, stream>>>(m->w, m->layout, f, x, k, mask, context, dev_table, n_steps, dt, u_jump,
                                                          seed, jet_offset, B, N);
    return cuda_ok(cudaGetLastError(), "generate_fp32 launch");
}

}  // namespace mmb
