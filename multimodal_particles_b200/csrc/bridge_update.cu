// bridge_update.cu — the fused, HBM-bound hybrid update (SURVEY.md §8a A8/A9/A11).
//
// One pass over the state: absorbing birth -> Euler step on (pT, eta, phi) -> telegraph jump on the
// token, all from registers.  Algorithmic traffic per particle-step (Dc=3, S=8): x r+w 24 B, v 12 B,
// logits 32 B, one jump uniform 4 B, token r+w 2 B, mask r 1 B = 75 B (84 B with the absorbing
// logit, its uniform and the mask write).  No data is reused, so there is nothing to stage in
// shared memory: each thread owns TWO consecutive particles, which makes every global access an
// 8- or 16-byte vector (x/v: 3 x float2, logits: S/2 x float4, u: float2) or a 2-byte word (tokens,
// masks), fully coalesced, with all loads issued before the first use.
#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

// particles per thread and CTAs per SM of the vector kernel: the variant with the highest bandwidth
// at 32 768 jets and more in profiles/r01_update_variants.md
constexpr int kPPT = 2;
constexpr int kUpdateMinBlocks = 5;

// NF consecutive floats -> registers with the widest aligned vector (16 B when NF % 4 == 0, else 8 B)
template <int NF, bool STREAM>
__device__ __forceinline__ void load_floats(const float* __restrict__ p, float (&out)[NF]) {
    if constexpr (NF % 4 == 0) {
#pragma unroll
        for (int i = 0; i < NF / 4; ++i) {
            const float4 q = STREAM ? __ldcs(reinterpret_cast<const float4*>(p) + i) : reinterpret_cast<const float4*>(p)[i];
            out[4 * i] = q.x; out[4 * i + 1] = q.y; out[4 * i + 2] = q.z; out[4 * i + 3] = q.w;
        }
    } else if constexpr (NF % 2 == 0) {
#pragma unroll
        for (int i = 0; i < NF / 2; ++i) {
            const float2 q = STREAM ? __ldcs(reinterpret_cast<const float2*>(p) + i) : reinterpret_cast<const float2*>(p)[i];
            out[2 * i] = q.x; out[2 * i + 1] = q.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < NF; ++i) out[i] = STREAM ? __ldcs(p + i) : p[i];
    }
}

template <int NF>
__device__ __forceinline__ void store_floats(float* __restrict__ p, const float (&v)[NF]) {
    if constexpr (NF % 4 == 0) {
#pragma unroll
        for (int i = 0; i < NF / 4; ++i)
            reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else if constexpr (NF % 2 == 0) {
#pragma unroll
        for (int i = 0; i < NF / 2; ++i) reinterpret_cast<float2*>(p)[i] = make_float2(v[2 * i], v[2 * i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < NF; ++i) p[i] = v[i];
    }
}

template <int PPT>
__device__ __forceinline__ void load_bytes(const uint8_t* __restrict__ p, int (&out)[PPT]) {
    if constexpr (PPT == 4) {
        const uchar4 q = *reinterpret_cast<const uchar4*>(p);
        out[0] = q.x; out[1] = q.y; out[2] = q.z; out[3] = q.w;
    } else if constexpr (PPT == 2) {
        const uchar2 q = *reinterpret_cast<const uchar2*>(p);
        out[0] = q.x; out[1] = q.y;
    } else {
        out[0] = *p;
    }
}

template <int PPT>
__device__ __forceinline__ void store_bytes(uint8_t* __restrict__ p, const int (&v)[PPT]) {
    if constexpr (PPT == 4) *reinterpret_cast<uchar4*>(p) = make_uchar4(v[0], v[1], v[2], v[3]);
    else if constexpr (PPT == 2) *reinterpret_cast<uchar2*>(p) = make_uchar2(v[0], v[1]);
    else *p = (uint8_t)v[0];
}

// PPT uniforms of consecutive particles drawn in the kernel: Philox keyed by (seed, global jet, stream, step, particle) exactly
// as mmb_philox_uniforms writes them (one block serves four consecutive particles of a jet)
template <int PPT>
__device__ __forceinline__ void draw_uniforms(const UpdateDraws& d, int stream_id, size_t first, float (&u)[PPT]) {
    const size_t jet = first / (size_t)d.N;
    const int n0 = (int)(first - jet * (size_t)d.N);
    if ((n0 & 3) + PPT <= 4 && n0 + PPT <= d.N) {   // all in one Philox block of one jet
        const uint4 r = philox_block(d.seed, d.jet_offset + jet, stream_id, d.step, n0 >> 2);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < PPT; ++j) u[j] = u01(w[(n0 & 3) + j]);
    } else {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            const size_t p = first + j, jj = p / (size_t)d.N;
            u[j] = philox_uniform(d.seed, d.jet_offset + jj, stream_id, d.step, (int)(p - jj * (size_t)d.N));
        }
    }
}

// Dc = 3.  Each thread owns PPT consecutive particles; group g covers particles [g*PPT, (g+1)*PPT).
template <int S>
__global__ void __launch_bounds__(256, kUpdateMinBlocks)
bridge_update_vec_kernel(float* __restrict__ x, uint8_t* __restrict__ k, uint8_t* __restrict__ mask,
                         const float* __restrict__ v, const float* __restrict__ logits,
                         const float* __restrict__ absorb, const float* __restrict__ uj,
                         const float* __restrict__ ua, StepScalars sc, size_t groups, int flags, UpdateDraws draws) {
    constexpr int PPT = kPPT;
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= groups) return;
    const bool do_euler = !(flags & MMB_FLAG_NO_EULER), do_jump = !(flags & MMB_FLAG_NO_JUMP),
               do_birth = (flags & MMB_FLAG_ABSORBING) != 0;

    // ---- all loads first: independent, 75*PPT bytes in flight per thread
    float xs[3 * PPT], vs[3 * PPT], lg[S * PPT], u[PPT], a[PPT], ub[PPT];
    int m[PPT], kk[PPT];
    load_bytes<PPT>(mask + g * PPT, m);
    if (do_euler) {
        load_floats<3 * PPT, false>(x + g * 3 * PPT, xs);
        load_floats<3 * PPT, true>(v + g * 3 * PPT, vs);
    }
    if (do_jump) {
        load_bytes<PPT>(k + g * PPT, kk);
        if (uj) load_floats<PPT, true>(uj + g * PPT, u);
        load_floats<S * PPT, true>(logits + g * S * PPT, lg);
    }
    if (do_birth) {
        load_floats<PPT, true>(absorb + g * PPT, a);
        if (ua) load_floats<PPT, true>(ua + g * PPT, ub);
    }
    if (do_jump && !uj) draw_uniforms<PPT>(draws, 0, g * PPT, u);       // under the loads in flight
    if (do_birth && !ua) draw_uniforms<PPT>(draws, 1, g * PPT, ub);
    // ---- birth (bridges.py:260-286)
    if (do_birth) {
#pragma unroll
        for (int j = 0; j < PPT; ++j) m[j] = absorbing_birth(m[j], a[j], ub[j], sc);
        store_bytes<PPT>(mask + g * PPT, m);
    }
    // ---- Euler (bridges.py:38-45)
    if (do_euler) {
#pragma unroll
        for (int i = 0; i < 3 * PPT; ++i) xs[i] = euler(xs[i], vs[i], sc.dt, (float)m[i / 3]);
        store_floats<3 * PPT>(x + g * 3 * PPT, xs);
    }
    // ---- telegraph jump (bridges.py:106-132,179-201)
    if (do_jump) {
        int nk[PPT];
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            float l[S];
#pragma unroll
            for (int s = 0; s < S; ++s) l[s] = lg[j * S + s];
            nk[j] = telegraph_jump<S>(l, kk[j], u[j], sc) * m[j];
        }
        store_bytes<PPT>(k + g * PPT, nk);
    }
}

// any Dc <= 8, S <= 32, any alignment: one particle per thread
__global__ void __launch_bounds__(256)
bridge_update_generic_kernel(float* __restrict__ x, uint8_t* __restrict__ k, uint8_t* __restrict__ mask,
                             const float* __restrict__ v, const float* __restrict__ logits,
                             const float* __restrict__ absorb, const float* __restrict__ uj,
                             const float* __restrict__ ua, StepScalars sc, size_t first, size_t count,
                             int Dc, int S, int flags, UpdateDraws draws) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const size_t p = first + i;
    int m = mask[p];
    float u1[1];
    if (flags & MMB_FLAG_ABSORBING) {
        if (ua) u1[0] = ua[p]; else draw_uniforms<1>(draws, 1, p, u1);
        m = absorbing_birth(m, absorb[p], u1[0], sc);
        mask[p] = (uint8_t)m;
    }
    if (!(flags & MMB_FLAG_NO_EULER))
        for (int c = 0; c < Dc; ++c) x[p * Dc + c] = euler(x[p * Dc + c], v[p * Dc + c], sc.dt, (float)m);
    if (!(flags & MMB_FLAG_NO_JUMP)) {
        if (uj) u1[0] = uj[p]; else draw_uniforms<1>(draws, 0, p, u1);
        k[p] = (uint8_t)(telegraph_jump_rt(logits + p * S, S, k[p], u1[0], sc) * m);
    }
}

static bool aligned16(const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int launch_bridge_update(float* x, uint8_t* k, uint8_t* mask, const float* v, const float* logits,
                         const float* absorb, const float* uj, const float* ua, StepScalars sc,
                         size_t P, int Dc, int S, int flags, cudaStream_t stream, const UpdateDraws* draws_in) {
    const UpdateDraws draws = draws_in ? *draws_in : UpdateDraws{0, 0, 0, 1};
    if (!draws_in && ((!(flags & MMB_FLAG_NO_JUMP) && !uj) || ((flags & MMB_FLAG_ABSORBING) && !ua)))
        return fail(MMB_EINVAL, "bridge update: uniforms missing");
    size_t done = 0;
    const bool vec_ok = Dc == 3 && (S == 8 || S == 4 || (flags & MMB_FLAG_NO_JUMP)) && aligned16(x) && aligned16(v) &&
                        aligned16(logits) && aligned16(absorb) && aligned16(uj) && aligned16(ua) &&
                        (reinterpret_cast<uintptr_t>(k) & 3u) == 0 && (reinterpret_cast<uintptr_t>(mask) & 3u) == 0;
    if (vec_ok && P >= 4) {
        const size_t groups = P / kPPT;
        const unsigned grid = (unsigned)((groups + 255) / 256);
        if (S == 4 && !(flags & MMB_FLAG_NO_JUMP))
            bridge_update_vec_kernel<4><<<grid, 256, 0, stream>>>(x, k, mask, v, logits, absorb, uj, ua, sc, groups, flags, draws);
        else
            bridge_update_vec_kernel<8><<<grid, 256, 0, stream>>>(x, k, mask, v, logits, absorb, uj, ua, sc, groups, flags, draws);
        done = groups * kPPT;
    }
    if (done < P) {
        const size_t count = P - done;
        const unsigned grid = (unsigned)((count + 255) / 256);
        bridge_update_generic_kernel<<<grid, 256, 0, stream>>>(x, k, mask, v, logits, absorb, uj, ua, sc, done, count, Dc, S, flags, draws);
    }
    return cuda_ok(cudaGetLastError(), "bridge_update launch");
}

// ---- uniforms exactly as the generation kernels draw them (tests) ------------------------------
__global__ void philox_uniforms_kernel(float* u, uint64_t seed, uint64_t jet_offset, int stream_id, int step0, int n_steps, int B, int N) {
    const size_t total = (size_t)n_steps * B * N;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int n = (int)(i % N);
        const int b = (int)((i / N) % B);
        const int s = (int)(i / ((size_t)N * B));
        u[i] = philox_uniform(seed, jet_offset + (uint64_t)b, stream_id, step0 + s, n);
    }
}

int launch_philox_uniforms(float* u, uint64_t seed, uint64_t jet_offset, int stream_id, int step0, int n_steps, int B, int N,
                           cudaStream_t stream) {
    const size_t total = (size_t)n_steps * B * N;
    if (total == 0) return MMB_OK;
    const unsigned grid = (unsigned)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
    philox_uniforms_kernel<<<grid, 256, 0, stream>>>(u, seed, jet_offset, stream_id, step0, n_steps, B, N);
    return cuda_ok(cudaGetLastError(), "philox_uniforms launch");
}

// ---- the three implementations of the jump rule on IDENTICAL logits and uniforms (tests) ----------------------------------
template <int S>
__global__ void __launch_bounds__(256) jump_variants_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ k,
                                                            const float* __restrict__ u, StepScalars sc, size_t P,
                                                            uint8_t* __restrict__ out_exact, uint8_t* __restrict__ out_tc,
                                                            uint8_t* __restrict__ out_mma) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (size_t)gridDim.x * blockDim.x) {
        float lg[S];
#pragma unroll
        for (int s = 0; s < S; ++s) lg[s] = __ldg(logits + i * S + s);
        const int kk = k[i];
        const float uu = __ldg(u + i);
        out_exact[i] = (uint8_t)telegraph_jump<S>(lg, kk, uu, sc);
        out_tc[i] = (uint8_t)telegraph_jump_fast<S>(lg, kk, uu, sc);
        out_mma[i] = (uint8_t)telegraph_jump_fast_ex2<S>(lg, kk, uu, sc.dt, sc.bc, sc.cc);
    }
}

int launch_jump_variants(const float* logits, const uint8_t* k, const float* u, StepScalars sc, size_t P, int S, uint8_t* out_exact,
                         uint8_t* out_tc, uint8_t* out_mma, cudaStream_t stream) {
    if (P == 0) return MMB_OK;
    const unsigned grid = (unsigned)((P + 255) / 256 < 148 * 16 ? (P + 255) / 256 : 148 * 16);
    if (S == 8) jump_variants_kernel<8><<<grid, 256, 0, stream>>>(logits, k, u, sc, P, out_exact, out_tc, out_mma);
    else if (S == 4) jump_variants_kernel<4><<<grid, 256, 0, stream>>>(logits, k, u, sc, P, out_exact, out_tc, out_mma);
    else return fail(MMB_EINVAL, "mmb_jump_variants: S must be 4 or 8 (the shapes the tensor-core engines are built for)");
    return cuda_ok(cudaGetLastError(), "jump_variants launch");
}

}  // namespace mmb
