// mmb_device.cuh — device helpers shared by the libmmbridge kernels (sm_100a).
//
// Everything on the fp32 path is spelled with round-to-nearest intrinsics (__fmaf_rn, __fmul_rn,
// __fadd_rn, __fdiv_rn) so that nvcc can neither contract nor reorder it: the fp32 kernels are
// bit-identical to oracle/mmb_oracle.c, which performs the same IEEE operations in the same order.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mmb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// named barrier `id` over `threads` threads (a multiple of 32)
__device__ __forceinline__ void named_bar(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// exp() from IEEE fp32 operations only (Cody-Waite + polynomial): the same function on CPU and GPU.
__device__ __forceinline__ float expf_exact(float x) {
    if (x != x) return x;
    if (x < -87.0f) return 0.0f;
    if (x > 88.0f) return __int_as_float(0x7f800000);
    float n = rintf(__fmul_rn(x, 1.44269504f));
    float r = __fmaf_rn(n, -0.693359375f, x);
    r = __fmaf_rn(n, 2.12194440e-4f, r);
    float p = 1.9875691500e-4f;
    p = __fmaf_rn(p, r, 1.3981999507e-3f);
    p = __fmaf_rn(p, r, 8.3334519073e-3f);
    p = __fmaf_rn(p, r, 4.1665795894e-2f);
    p = __fmaf_rn(p, r, 1.6666665459e-1f);
    p = __fmaf_rn(p, r, 5.0000001201e-1f);
    float r2 = __fmul_rn(r, r);
    float y = __fadd_rn(__fmaf_rn(p, r2, r), 1.0f);
    int e = (int)n;
    return __fmul_rn(y, __int_as_float((e + 127) << 23));
}

// expf_exact with gradual underflow below 2^-126 (mmbo_expf_dn): the batch-axis softmax of the trans-dimensional token rule
__device__ __forceinline__ float expf_exact_dn(float x) {
    if (!(x < -87.0f)) return expf_exact(x);
    if (x < -104.0f) return 0.0f;
    float n = rintf(__fmul_rn(x, 1.44269504f));
    float r = __fmaf_rn(n, -0.693359375f, x);
    r = __fmaf_rn(n, 2.12194440e-4f, r);
    float p = 1.9875691500e-4f;
    p = __fmaf_rn(p, r, 1.3981999507e-3f);
    p = __fmaf_rn(p, r, 8.3334519073e-3f);
    p = __fmaf_rn(p, r, 4.1665795894e-2f);
    p = __fmaf_rn(p, r, 1.6666665459e-1f);
    p = __fmaf_rn(p, r, 5.0000001201e-1f);
    float r2 = __fmul_rn(r, r);
    float y = __fadd_rn(__fmaf_rn(p, r2, r), 1.0f);
    int e = (int)n + 64;
    return __fmul_rn(__fmul_rn(y, __int_as_float((e + 127) << 23)), 5.42101086e-20f);
}

// packed fp32 pair arithmetic (sm_100 FFMA2 / FADD2 / FMUL2): two IEEE fp32 operations per issue slot
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b0, float b1, float c0, float c1) {
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d0), "=f"(d1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
}
__device__ __forceinline__ void fadd2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d0), "=f"(d1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
__device__ __forceinline__ void fmul2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d0), "=f"(d1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}

__device__ __forceinline__ float lrelu(float a) { return a > 0.0f ? a : __fmul_rn(a, 0.01f); }
// the tensor-core engines' branch-free form
__device__ __forceinline__ float lrelu_fast(float a) { return fmaxf(a, 0.01f * a); }

__device__ __forceinline__ float selu(float a) {
    const float scale = 1.0507009873554804934193349852946f;
    const float alpha_scale = 1.0507009873554804934193349852946f * 1.6732632423543772848170429916717f;
    return a > 0.0f ? __fmul_rn(scale, a) : __fmul_rn(alpha_scale, __fadd_rn(expf_exact(a), -1.0f));
}

// Philox4x32-10; counter = (n>>2, step, jet_lo, jet_hi*4 + stream), key = seed.  One call serves
// four consecutive particles.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ float u01(uint32_t bits) { return (float)(bits >> 8) * (1.0f / 16777216.0f); }

__device__ __forceinline__ uint4 philox_block(uint64_t seed, uint64_t jet, int stream_id, int step, int n4) {
    return philox4x32_10(make_uint4((uint32_t)n4, (uint32_t)step, (uint32_t)jet,
                                    (uint32_t)(jet >> 32) * 4u + (uint32_t)stream_id),
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}

__device__ __forceinline__ float philox_uniform(uint64_t seed, uint64_t jet, int stream_id, int step, int n) {
    const uint4 r = philox_block(seed, jet, stream_id, step, n >> 2);
    const uint32_t w = (n & 3) == 0 ? r.x : (n & 3) == 1 ? r.y : (n & 3) == 2 ? r.z : r.w;
    return u01(w);
}

// Scalars of one solver step (MmbStepTable row).
struct StepScalars {
    float dt, bc, cc, sp;
};

// The hybrid update of one particle — the device twin of update_particle() in oracle/mmb_oracle.c
// (bridges.py:260-286, 38-45, 106-132, 179-201; Form B categorical, SURVEY.md §A.4).
// `logits` / `x` / `v` are per-particle register arrays.
template <int S>
__device__ __forceinline__ int telegraph_jump(const float (&lg)[S], int k, float u, const StepScalars& sc) {
    float mx = lg[0];
#pragma unroll
    for (int s = 1; s < S; ++s) mx = lg[s] > mx ? lg[s] : mx;
    float e[S], z = 0.0f;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        e[s] = expf_exact(__fadd_rn(lg[s], -mx));
        z = __fadd_rn(z, e[s]);
    }
    const float zinv = __fdiv_rn(1.0f, z);
    float ek = e[0];
#pragma unroll
    for (int s = 1; s < S; ++s) ek = (k == s) ? e[s] : ek;
    const float ck = __fmul_rn(sc.cc, __fmul_rn(ek, zinv));
    float lam[S], Lam = 0.0f;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const float rate = __fadd_rn(__fadd_rn(1.0f, __fmul_rn(sc.bc, __fmul_rn(e[s], zinv))), ck);
        lam[s] = __fmul_rn(rate, sc.dt);
        Lam = __fadd_rn(Lam, lam[s]);
    }
    const float E = expf_exact(-Lam);
    int nk = k;
    float c = 0.0f;
    bool open = true;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        c = __fadd_rn(c, __fmul_rn(lam[s], E));
        if (open && u < c) { nk = s; open = false; }
    }
    return nk;
}

// runtime-S variant (S <= 32), logits read through a pointer (global or shared)
__device__ __forceinline__ int telegraph_jump_rt(const float* lg, int S, int k, float u, const StepScalars& sc) {
    float mx = lg[0];
    for (int s = 1; s < S; ++s) mx = lg[s] > mx ? lg[s] : mx;
    float z = 0.0f;
    for (int s = 0; s < S; ++s) z = __fadd_rn(z, expf_exact(__fadd_rn(lg[s], -mx)));
    const float zinv = __fdiv_rn(1.0f, z);
    const float ck = __fmul_rn(sc.cc, __fmul_rn(expf_exact(__fadd_rn(lg[k], -mx)), zinv));
    float Lam = 0.0f;
    for (int s = 0; s < S; ++s) {
        const float q = __fmul_rn(expf_exact(__fadd_rn(lg[s], -mx)), zinv);
        Lam = __fadd_rn(Lam, __fmul_rn(__fadd_rn(__fadd_rn(1.0f, __fmul_rn(sc.bc, q)), ck), sc.dt));
    }
    const float E = expf_exact(-Lam);
    float c = 0.0f;
    for (int s = 0; s < S; ++s) {
        const float q = __fmul_rn(expf_exact(__fadd_rn(lg[s], -mx)), zinv);
        const float lam = __fmul_rn(__fadd_rn(__fadd_rn(1.0f, __fmul_rn(sc.bc, q)), ck), sc.dt);
        c = __fadd_rn(c, __fmul_rn(lam, E));
        if (u < c) return s;
    }
    return k;
}


// ---- the jump rule of the tensor-core engines -----------------------------------------------------------------------------
// Same categorical (Form B) as telegraph_jump above, evaluated with fast intrinsics and without branches: the logits of those
// engines already carry 16-bit operand rounding, so the exact-exp contract of the fp32 path buys nothing there.  Given
// IDENTICAL logits the variants can disagree with the exact rule only when the uniform lies within rounding of a threshold;
// tests/test_gpu_jump.py feeds all three the same 5*10^7 draws and lists every disagreement with its distance to the threshold.
__device__ __forceinline__ float ex2_fast(float a) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    return r;
}

// tcgen05 engine (epic_tc.cu)
template <int S>
__device__ __forceinline__ int telegraph_jump_fast(const float (&lg)[S], int k, float u, const StepScalars& sc) {
    float mx = lg[0];
#pragma unroll
    for (int s = 1; s < S; ++s) mx = fmaxf(mx, lg[s]);
    float e[S], z = 0.0f, ek = 0.0f;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        e[s] = __expf(lg[s] - mx);
        z += e[s];
        ek = (k == s) ? e[s] : ek;
    }
    const float zinv = __fdividef(1.0f, z);
    const float base = (1.0f + sc.cc * ek * zinv) * sc.dt, slope = sc.bc * zinv * sc.dt;
    float lam[S], Lam = 0.0f;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        lam[s] = fmaf(e[s], slope, base);
        Lam += lam[s];
    }
    const float E = __expf(-Lam);
    float c = 0.0f;
    int below = 0;  // number of thresholds c_s <= u  ==  index of the first s with u < c_s
#pragma unroll
    for (int s = 0; s < S; ++s) {
        c = fmaf(lam[s], E, c);
        below += (u >= c) ? 1 : 0;
    }
    return below < S ? below : k;
}


// warp-MMA engine (epic_mma.cu): exp2 with pre-scaled arguments, Lambda in closed form (the softmax sums to one)
template <int S>
__device__ __forceinline__ int telegraph_jump_fast_ex2(const float (&lg)[S], int k, float u, float dt, float bc, float cc) {
    constexpr float kLog2e = 1.4426950408889634f;
    float mx = lg[0];
#pragma unroll
    for (int s = 1; s < S; ++s) mx = fmaxf(mx, lg[s]);
    const float nmx = -mx * kLog2e;
    float e[S], z = 0.0f, ek = 0.0f;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        e[s] = ex2_fast(fmaf(lg[s], kLog2e, nmx));
        z += e[s];
        ek = (k == s) ? e[s] : ek;
    }
    const float zinv = __fdividef(1.0f, z);
    const float base = fmaf(cc * ek, zinv, 1.0f) * dt, slope = bc * zinv * dt;
    const float Lam = fmaf((float)S, base, bc * dt);           // sum_s (base + slope e_s) = S base + slope z
    const float E = ex2_fast(-Lam * kLog2e);
    const float bE = base * E, sE = slope * E;
    float c = 0.0f;
    int below = 0;   // number of thresholds c_s <= u  ==  index of the first s with u < c_s
#pragma unroll
    for (int s = 0; s < S; ++s) {
        c += fmaf(e[s], sE, bE);
        below += (u >= c) ? 1 : 0;
    }
    return below < S ? below : k;
}


__device__ __forceinline__ int absorbing_birth(int m, float a, float u, const StepScalars& sc) {
    const float sg = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf_exact(-a)));
    float p = __fmul_rn(sc.dt, __fmul_rn(sc.sp, sg));
    p = p > 1.0f ? 1.0f : p;
    const int born = (u < p) ? 1 : 0;
    return (m == 1) ? 1 : born;
}

__device__ __forceinline__ float euler(float x, float v, float dt, float mf) {
    return __fmul_rn(__fadd_rn(x, __fmul_rn(dt, v)), mf);
}

// The loss terms of one live particle (mbm.py:167-197): the squared error of its drift v against x1 - x0 over Dc components,
// and its cross entropy max + log sum exp - logits[k1].  Shared by the bridge losses and the loss-gradient kernel.
// Plain loads, not __ldg: the loss-gradient kernel passes rows it wrote earlier in the same launch.
__device__ __forceinline__ float2 bridge_loss_terms(const float* v, const float* x0, const float* x1, int Dc, const float* logits,
                                                    int S, int k1) {
    float e = 0.0f;
    for (int c = 0; c < Dc; ++c) {
        const float d = v[c] - (x1[c] - x0[c]);
        e = fmaf(d, d, e);
    }
    float mx = -INFINITY;
    for (int s = 0; s < S; ++s) mx = fmaxf(mx, logits[s]);
    float se = 0.0f;
    for (int s = 0; s < S; ++s) se += expf(logits[s] - mx);
    return make_float2(e, (mx + logf(se)) - logits[k1]);
}

}  // namespace mmb
