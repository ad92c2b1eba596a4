// bridge_sample.cu — the forward half of a training / validation step (SURVEY.md §8f N2): conditional bridge sampling and the
// masked losses.  Both are single-pass, HBM-bound kernels.
//
// Reference (mp/ = /root/reference/multimodal_particles/):
//   MultiModalBridgeMatching.sample_bridges      mp/models/generative/multimodal_bridge_matching.py:148-165
//   LinearUniformBridge.sample                   mp/models/generative/bridges.py:23-27
//   TelegraphBridge.sample / transition_probability / conditional_probability   bridges.py:99-104,134-177
//   AbsorbingBridge.sample                       bridges.py:233-249
//   loss_continuous / loss_discrete              multimodal_bridge_matching.py:167-197
#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {
namespace {

// x_t = (t x1 + (1-t) x0) + sigma z;  k_t ~ Categorical(P(k | k0, k1, t)) by inverse CDF on one uniform.
// One thread per particle; same IEEE operations in the same order as oracle/mmb_oracle.c (bit-identical with injected draws).
__global__ void __launch_bounds__(256) sample_bridges_kernel(const float* __restrict__ x0, const float* __restrict__ x1,
                                                             const uint8_t* __restrict__ k0, const uint8_t* __restrict__ k1,
                                                             const float* __restrict__ ts, float sigma, float neg_s_gamma, int S,
                                                             const float* __restrict__ z, const float* __restrict__ u, uint64_t seed,
                                                             uint64_t jet_offset, int B, int N, float* __restrict__ xt,
                                                             uint8_t* __restrict__ kt) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * N) return;
    const int b = (int)(i / N), n = (int)(i % N);
    const float t = __ldg(ts + b), omt = __fadd_rn(1.0f, -t);
    float zz[3], uu;
    if (z) {
        zz[0] = __ldg(z + i * 3); zz[1] = __ldg(z + i * 3 + 1); zz[2] = __ldg(z + i * 3 + 2);
        uu = __ldg(u + i);
    } else {   // ONE Philox block (stream 12) per particle: the top 24 bits of its words feed Box-Muller (three normals), the low
               // bytes of x, y, z make the 24-bit uniform of the token draw
        const uint4 r = philox_block(seed, jet_offset + (uint64_t)b, 12, 0, n);
        const float u1 = ((float)(r.x >> 8) + 1.0f) * (1.0f / 16777216.0f), u2 = (float)(r.y >> 8) * (1.0f / 16777216.0f);
        const float rad = sqrtf(-2.0f * __logf(u1));
        float sn, cs;
        __sincosf(6.283185307179586f * u2, &sn, &cs);
        zz[0] = rad * cs; zz[1] = rad * sn;
        const float u3 = ((float)(r.z >> 8) + 1.0f) * (1.0f / 16777216.0f), u4 = (float)(r.w >> 8) * (1.0f / 16777216.0f);
        zz[2] = sqrtf(-2.0f * __logf(u3)) * __cosf(6.283185307179586f * u4);
        uu = (float)((r.x & 0xffu) | ((r.y & 0xffu) << 8) | ((r.z & 0xffu) << 16)) * (1.0f / 16777216.0f);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float lin = __fadd_rn(__fmul_rn(t, __ldg(x1 + i * 3 + c)), __fmul_rn(omt, __ldg(x0 + i * 3 + c)));
        xt[i * 3 + c] = __fadd_rn(lin, __fmul_rn(sigma, zz[c]));
    }
    // telegraph bridge posterior (bridges.py:134-177): p(a -> b; dt) = 1/S + w(dt) (-1/S + [a == b]),  w = exp(-S gamma dt)
    const float inv_s = __fdiv_rn(1.0f, (float)S), ninv_s = __fdiv_rn(-1.0f, (float)S);
    // the three exponentials depend on the jet alone: when a warp lies inside one jet, three lanes compute one each
    float w1, w0, w01;
    {
        const float arg1 = __fmul_rn(neg_s_gamma, __fadd_rn(1.0f, -t));   // k -> k1 over [t, 1]
        const float arg0 = __fmul_rn(neg_s_gamma, __fadd_rn(t, -0.0f));   // k0 -> k over [0, t]
        const float arg01 = __fmul_rn(neg_s_gamma, 1.0f);                 // k0 -> k1 over [0, 1]
        if ((N & 31) == 0) {   // B * N is then a multiple of 32 as well: every lane of the warp is here, all on jet b
            const int lane = threadIdx.x & 31;
            const float mine = expf_exact(lane == 0 ? arg1 : (lane == 1 ? arg0 : arg01));
            w1 = __shfl_sync(0xffffffffu, mine, 0);
            w0 = __shfl_sync(0xffffffffu, mine, 1);
            w01 = __shfl_sync(0xffffffffu, mine, 2);
        } else {
            w1 = expf_exact(arg1); w0 = expf_exact(arg0); w01 = expf_exact(arg01);
        }
    }
    const int a0 = k0[i], a1 = k1[i];
    const float p01 = __fadd_rn(inv_s, __fmul_rn(w01, __fadd_rn(ninv_s, a0 == a1 ? 1.0f : 0.0f)));
    // P(k) ~ pa(k) pb(k) / p01 takes three values: at k = k1, at k = k0, elsewhere (k0 = k1: two).  Same IEEE operations on the
    // same operands as the per-k loop of the oracle, evaluated once per distinct value; the sums run over k in order.
    const float pa_hit = __fadd_rn(inv_s, __fmul_rn(w1, __fadd_rn(ninv_s, 1.0f))), pa_miss = __fadd_rn(inv_s, __fmul_rn(w1, __fadd_rn(ninv_s, 0.0f)));
    const float pb_hit = __fadd_rn(inv_s, __fmul_rn(w0, __fadd_rn(ninv_s, 1.0f))), pb_miss = __fadd_rn(inv_s, __fmul_rn(w0, __fadd_rn(ninv_s, 0.0f)));
    const float t_else = __fdiv_rn(__fmul_rn(pa_miss, pb_miss), p01);
    const float t_k1 = __fdiv_rn(__fmul_rn(pa_hit, a0 == a1 ? pb_hit : pb_miss), p01);
    const float t_k0 = a0 == a1 ? t_k1 : __fdiv_rn(__fmul_rn(pa_miss, pb_hit), p01);
    float tot = 0.0f;
    for (int k = 0; k < S; ++k) tot = __fadd_rn(tot, k == a1 ? t_k1 : (k == a0 ? t_k0 : t_else));
    const float q_else = __fdiv_rn(t_else, tot), q_k1 = __fdiv_rn(t_k1, tot), q_k0 = a0 == a1 ? q_k1 : __fdiv_rn(t_k0, tot);
    int pick = S - 1;
    bool found = false;
    float c = 0.0f;
    for (int k = 0; k < S; ++k) {
        c = __fadd_rn(c, k == a1 ? q_k1 : (k == a0 ? q_k0 : q_else));
        if (!found && uu < c) { pick = k; found = true; }
    }
    kt[i] = (uint8_t)pick;
}

// mask_t = [u < SP(t)] | target_mask  (AbsorbingBridge.sample, bridges.py:233-249); sp[b] = survival probability of jet b's time.
// Four consecutive particles per thread when N % 4 == 0: one Philox block (stream 14, counter = n / 4) and one 4-byte load/store.
__global__ void __launch_bounds__(256) absorbing_sample_kernel(const float* __restrict__ sp, const uint8_t* __restrict__ target_mask,
                                                               const float* __restrict__ u, uint64_t seed, uint64_t jet_offset, int B, int N,
                                                               uint8_t* __restrict__ mask_t) {
    if ((N & 3) == 0) {
        const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x, i = q * 4;
        if (i >= (size_t)B * N) return;
        const int b = (int)(i / N), n = (int)(i % N);
        const float s = __ldg(sp + b);
        float uu[4];
        if (u) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(u + i));
            uu[0] = v.x; uu[1] = v.y; uu[2] = v.z; uu[3] = v.w;
        } else {
            const uint4 r = philox_block(seed, jet_offset + (uint64_t)b, 14, 0, n >> 2);
            uu[0] = u01(r.x); uu[1] = u01(r.y); uu[2] = u01(r.z); uu[3] = u01(r.w);
        }
        const uchar4 tm = *reinterpret_cast<const uchar4*>(target_mask + i);
        uchar4 o;
        o.x = (tm.x || uu[0] < s) ? 1 : 0; o.y = (tm.y || uu[1] < s) ? 1 : 0;
        o.z = (tm.z || uu[2] < s) ? 1 : 0; o.w = (tm.w || uu[3] < s) ? 1 : 0;
        *reinterpret_cast<uchar4*>(mask_t + i) = o;
        return;
    }
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * N) return;
    const int b = (int)(i / N), n = (int)(i % N);
    const float uu = u ? __ldg(u + i) : philox_uniform(seed, jet_offset + (uint64_t)b, 14, 0, n);   // word n & 3 of the quad's block, like the vector branch
    mask_t[i] = (target_mask[i] || uu < __ldg(sp + b)) ? 1 : 0;
}

// masked MSE (drift matching) and cross entropy, summed: stage 1 writes one (mse, ce, count) triple per block in a fixed order,
// stage 2 adds the triples sequentially -> deterministic sums
constexpr int kLossThreads = 256;
__global__ void __launch_bounds__(kLossThreads) bridge_losses_partial_kernel(const float* __restrict__ v, const float* __restrict__ logits,
                                                                             const float* __restrict__ x0, const float* __restrict__ x1,
                                                                             const uint8_t* __restrict__ k1, const uint8_t* __restrict__ mask,
                                                                             size_t P, int S, float* __restrict__ partial) {
    __shared__ float s_red[3][kLossThreads / 32];
    float mse = 0.0f, ce = 0.0f, cnt = 0.0f;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (size_t)gridDim.x * blockDim.x) {
        if (!mask[i]) continue;
        const float2 t = bridge_loss_terms(v + i * 3, x0 + i * 3, x1 + i * 3, 3, logits + i * S, S, k1[i]);
        mse += t.x;
        ce += t.y;
        cnt += 1.0f;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        mse += __shfl_xor_sync(0xffffffffu, mse, o);
        ce += __shfl_xor_sync(0xffffffffu, ce, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = mse; s_red[1][threadIdx.x >> 5] = ce; s_red[2][threadIdx.x >> 5] = cnt; }
    __syncthreads();
    if (threadIdx.x < 3) {
        float a = 0.0f;
        for (int w = 0; w < kLossThreads / 32; ++w) a += s_red[threadIdx.x][w];
        partial[(size_t)blockIdx.x * 3 + threadIdx.x] = a;
    }
}
__global__ void bridge_losses_final_kernel(const float* __restrict__ partial, int n_blocks, float* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double m = 0, c = 0, n = 0;
        for (int i = 0; i < n_blocks; ++i) { m += partial[i * 3]; c += partial[i * 3 + 1]; n += partial[i * 3 + 2]; }
        out[0] = (float)(m / n); out[1] = (float)(c / n); out[2] = (float)n;
    }
}

}  // namespace

int launch_sample_bridges(const float* x0, const float* x1, const uint8_t* k0, const uint8_t* k1, const float* ts, float sigma, float gamma,
                          int S, const float* z, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N, float* xt, uint8_t* kt,
                          cudaStream_t stream) {
    const size_t P = (size_t)B * N;
    const float neg_s_gamma = (float)(-(double)S * (double)gamma);
    sample_bridges_kernel<<<(unsigned)((P + 255) / 256), 256, 0, stream>>>(x0, x1, k0, k1, ts, sigma, neg_s_gamma, S, z, u, seed, jet_offset, B, N,
                                                                           xt, kt);
    return cuda_ok(cudaGetLastError(), "sample_bridges launch");
}

int launch_absorbing_sample(const float* sp, const uint8_t* target_mask, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N,
                            uint8_t* mask_t, cudaStream_t stream) {
    const size_t P = (N & 3) == 0 ? (size_t)B * N / 4 : (size_t)B * N;   // threads: four particles each when N % 4 == 0
    absorbing_sample_kernel<<<(unsigned)((P + 255) / 256), 256, 0, stream>>>(sp, target_mask, u, seed, jet_offset, B, N, mask_t);
    return cuda_ok(cudaGetLastError(), "absorbing_sample launch");
}

int bridge_losses_blocks(size_t P) {
    const size_t want = (P + kLossThreads - 1) / kLossThreads;
    return (int)(want < 148 * 8 ? (want ? want : 1) : 148 * 8);
}

int launch_bridge_losses(const float* v, const float* logits, const float* x0, const float* x1, const uint8_t* k1, const uint8_t* mask,
                         size_t P, int S, float* out, float* partial, cudaStream_t stream) {
    const int blocks = bridge_losses_blocks(P);
    bridge_losses_partial_kernel<<<blocks, kLossThreads, 0, stream>>>(v, logits, x0, x1, k1, mask, P, S, partial);
    bridge_losses_final_kernel<<<1, 32, 0, stream>>>(partial, blocks, out);
    return cuda_ok(cudaGetLastError(), "bridge_losses launch");
}

}  // namespace mmb
