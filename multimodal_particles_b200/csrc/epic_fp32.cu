// epic_fp32.cu — the fp32 EPiC forward (epic_fp32.cuh) as the parity kernel and as the fused generation kernel, state in
// shared memory.
#include "epic_fp32.cuh"

namespace mmb {

namespace {

// shared-memory carve-up (floats)
__host__ __device__ inline size_t smem_floats(const Fp32Dims& f, int N) {
    return (size_t)(f.T + f.X) + f.H + (2 * f.H + f.G + f.T + f.X) + f.H + f.H + f.G + f.G + f.H + 4 * f.H + 8 +
           (size_t)N * f.HS * 2 + (size_t)N * f.RS;
}

__device__ inline Fp32Bufs carve(float* base, const Fp32Dims& f, int N) {
    Fp32Bufs s;
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

__global__ void __launch_bounds__(kFp32Threads)
epic_forward_fp32_kernel(const float* __restrict__ W, MmbEpicLayout Lo, Fp32Dims f,
                         const float* __restrict__ x, const uint8_t* __restrict__ k, const uint8_t* __restrict__ mask,
                         const float* __restrict__ temb, int temb_stride, int N,
                         float* __restrict__ v_out, float* __restrict__ logits_out, float* __restrict__ hidden_out) {
    extern __shared__ float smem[];
    const Fp32Bufs s = carve(smem, f, N);
    const size_t b = blockIdx.x;
    for (int i = threadIdx.x; i < f.T + f.X; i += kFp32Threads) s.temb[i] = temb[b * temb_stride + i];
    __syncthreads();
    epic_forward_jet(W, Lo, f, s, x + b * N * f.Dc, k + b * N, mask + b * N, N,
                     v_out + b * N * f.Dc, logits_out + b * N * f.S, hidden_out ? hidden_out + b * N * f.H : nullptr);
}

// Whole generation for one jet per CTA, state in shared memory across all steps
// (MultiModalBridgeMatching.simulate_dynamics, mbm.py:199-216).
__global__ void __launch_bounds__(kFp32Threads)
generate_fp32_kernel(const float* __restrict__ W, MmbEpicLayout Lo, Fp32Dims f,
                     float* __restrict__ x, uint8_t* __restrict__ k, const uint8_t* __restrict__ mask,
                     const float* __restrict__ context, const float* __restrict__ table, int n_steps, float dt,
                     const float* __restrict__ u_jump, uint64_t seed, uint64_t jet_offset, int B, int N) {
    extern __shared__ float smem[];
    const Fp32Bufs s = carve(smem, f, N);
    float* sx = smem + smem_floats(f, N);
    float* sv = sx + (size_t)N * f.Dc;
    float* slog = sv + (size_t)N * f.Dc;
    uint8_t* sk = reinterpret_cast<uint8_t*>(slog + (size_t)N * f.S);
    uint8_t* sm = sk + ((N + 15) & ~15);
    const size_t b = blockIdx.x;
    const int tid = threadIdx.x;
    for (int i = tid; i < N * f.Dc; i += kFp32Threads) sx[i] = x[b * N * f.Dc + i];
    for (int n = tid; n < N; n += kFp32Threads) { sk[n] = k[b * N + n]; sm[n] = mask[b * N + n]; }
    const float* temb_tab = table + (size_t)n_steps * 4;
    for (int i = tid; i < f.X; i += kFp32Threads) s.temb[f.T + i] = context[b * f.X + i];   // constant over the steps (mbm.py:143-144)
    for (int step = 0; step < n_steps; ++step) {
        for (int i = tid; i < f.T; i += kFp32Threads) s.temb[i] = temb_tab[(size_t)step * f.T + i];
        __syncthreads();
        epic_forward_jet(W, Lo, f, s, sx, sk, sm, N, sv, slog, nullptr);
        const StepScalars sc{dt, table[step * 4 + 0], table[step * 4 + 1], table[step * 4 + 2]};
        for (int n = tid; n < N; n += kFp32Threads) {   // each particle is read and written by its owner only
            const int m = sm[n];
            for (int c = 0; c < f.Dc; ++c) sx[n * f.Dc + c] = euler(sx[n * f.Dc + c], sv[n * f.Dc + c], dt, (float)m);
            const float u = u_jump ? u_jump[((size_t)step * B + b) * N + n]
                                   : philox_uniform(seed, jet_offset + b, 0, step, n);
            sk[n] = (uint8_t)(telegraph_jump_rt(slog + (size_t)n * f.S, f.S, sk[n], u, sc) * m);
        }
        __syncthreads();
    }
    for (int i = tid; i < N * f.Dc; i += kFp32Threads) x[b * N * f.Dc + i] = sx[i];
    for (int n = tid; n < N; n += kFp32Threads) k[b * N + n] = sk[n];
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
    epic_forward_fp32_kernel<<<B, kFp32Threads, bytes, stream>>>(m->w, m->layout, f, x, k, mask, temb, temb_stride, N,
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
    generate_fp32_kernel<<<B, kFp32Threads, bytes, stream>>>(m->w, m->layout, f, x, k, mask, context, dev_table, n_steps, dt, u_jump,
                                                              seed, jet_offset, B, N);
    return cuda_ok(cudaGetLastError(), "generate_fp32 launch");
}

}  // namespace mmb
