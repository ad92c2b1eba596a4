// jet_metrics.cu — the sample statistics behind the Fréchet and kernel physics distances (FPD, KPD) of Kansal et al.
// (arXiv:2211.10295), on rows the caller draws by index.  Definitions: include/mmbridge.h and DESIGN.md §4.6d.
//
// moments_kernel: one block per draw.  Rows are gathered (x * scale, exact in fp64) into a shared tile; each thread owns one
// entry of the sum or of the upper triangle of x x^T and a fixed residue class of the tile's rows, and the row lanes of an
// entry are added in lane order.
// kpd_strip_kernel: grid (row strips, term, batch).  A block holds one 64-row strip of the first sample in shared memory and
// walks the 64-row tiles of the second sample (b >= a for the two self terms, every b for the cross term), 4 x 4 pairs per
// thread, dot products and the polynomial kernel in fp64.  Each strip writes one fp64 partial; kpd_final_kernel adds the
// partials of each term in a fixed order.  Every shape is fixed by the arguments, so both are bit-identical from call to call.
#include "mmb_internal.h"

namespace mmb {

namespace {

constexpr int kMomThreads = 512;
constexpr int kMomTileElems = 4096;                                  // doubles of the gathered row tile
constexpr int kMomMaxItems = MMB_MET_MAX_D + MMB_MET_MAX_D * (MMB_MET_MAX_D + 1) / 2;
constexpr int kMomPerThread = (kMomMaxItems + kMomThreads - 1) / kMomThreads;
constexpr int kKpdThreads = 256;
constexpr int kKpdTile = 64;                                         // 16 x 16 threads, 4 x 4 pairs each
constexpr int kKpdFinalThreads = 256;

__device__ __forceinline__ double scaled(const float* x, long long ld, int row, int c, const float* scale) {
    const double v = (double)x[(long long)row * ld + c];
    return scale ? v * (double)scale[c] : v;   // the product of two floats is exact in fp64
}

// entry e of the moment list: e < d is sum(x_a); then the upper triangle of x x^T row by row, (a, b) with a <= b
__device__ __forceinline__ void moment_entry(int e, int d, int& a, int& b) {
    if (e < d) { a = e; b = -1; return; }
    e -= d;
    a = 0;
    while (e >= d - a) { e -= d - a; ++a; }
    b = a + e;
}

__global__ void __launch_bounds__(kMomThreads)
moments_kernel(const float* __restrict__ x, long long ldx, int d, const float* __restrict__ scale, const int* __restrict__ idx,
               int rows, double* __restrict__ sum, double* __restrict__ sumsq) {
    __shared__ double tile[kMomTileElems];
    __shared__ double red[kMomThreads];
    const int draw = blockIdx.x;
    const int items = d + d * (d + 1) / 2;
    const int lanes = items < kMomThreads ? kMomThreads / items : 1;   // row lanes per entry
    const int R = kMomTileElems / d < 256 ? kMomTileElems / d : 256;  // rows per tile
    const int* id = idx + (long long)draw * rows;
    int ea[kMomPerThread], eb[kMomPerThread], lane = 0, mine = 0;
    if (lanes > 1) {
        if (threadIdx.x < lanes * items) {
            moment_entry(threadIdx.x % items, d, ea[0], eb[0]);
            lane = threadIdx.x / items;
            mine = 1;
        }
    } else {
        for (int e = threadIdx.x; e < items; e += kMomThreads) moment_entry(e, d, ea[mine], eb[mine]), ++mine;
    }
    double acc[kMomPerThread];
#pragma unroll
    for (int k = 0; k < kMomPerThread; ++k) acc[k] = 0.0;
    for (int r0 = 0; r0 < rows; r0 += R) {
        const int nr = rows - r0 < R ? rows - r0 : R;
        __syncthreads();
        for (int e = threadIdx.x; e < nr * d; e += kMomThreads) {
            const int r = e / d, c = e - r * d;
            tile[e] = scaled(x, ldx, id[r0 + r], c, scale);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kMomPerThread; ++k) {
            if (k >= mine) break;
            const int a = ea[k], b = eb[k];
            double s = acc[k];
            if (b < 0)
                for (int r = lane; r < nr; r += lanes) s += tile[r * d + a];
            else
                for (int r = lane; r < nr; r += lanes) s += tile[r * d + a] * tile[r * d + b];
            acc[k] = s;
        }
    }
    if (lanes > 1) {
        red[threadIdx.x] = mine ? acc[0] : 0.0;
        __syncthreads();
        if (threadIdx.x < items) {
            double s = 0.0;
            for (int l = 0; l < lanes; ++l) s += red[l * items + threadIdx.x];
            acc[0] = s;
            mine = 1;
        } else {
            mine = 0;
        }
    }
    for (int k = 0; k < mine; ++k) {
        const int a = ea[k], b = eb[k];
        if (b < 0) {
            sum[(long long)draw * d + a] = acc[k];
        } else {
            double* S = sumsq + (long long)draw * d * d;
            S[a * d + b] = acc[k];
            S[b * d + a] = acc[k];
        }
    }
}

// gathered rows: g[batch][sample][B][d] fp64, sample 0 = real, 1 = gen
__global__ void kpd_gather_kernel(const float* __restrict__ real, long long ldr, const float* __restrict__ gen, long long ldg, int d,
                                  const float* __restrict__ scale, const int* __restrict__ idx_real, const int* __restrict__ idx_gen,
                                  int batches, int B, double* __restrict__ g) {
    const long long per = (long long)B * d, total = (long long)batches * 2 * per;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long bs = e / per, rc = e - bs * per;
        const int batch = (int)(bs >> 1), sample = (int)(bs & 1), r = (int)(rc / d), c = (int)(rc - (long long)r * d);
        const long long slot = (long long)batch * B + r;
        g[e] = sample ? scaled(gen, ldg, idx_gen[slot], c, scale) : scaled(real, ldr, idx_real[slot], c, scale);
    }
}

__device__ __forceinline__ double kpd_block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    return s;
}

// loads rows [r0, r0 + 64) of one gathered sample into t[64][ld], zeros past B
__device__ __forceinline__ void kpd_load(const double* __restrict__ src, int r0, int B, int d, int ld, double* t) {
    for (int e = threadIdx.x; e < kKpdTile * d; e += kKpdThreads) {
        const int r = e / d, c = e - r * d;
        t[r * ld + c] = r0 + r < B ? src[(long long)(r0 + r) * d + c] : 0.0;
    }
}

// partial[batch][term][a]: term 0 = sum_{i != j} k(r_i, r_j), 1 = the same over gen, 2 = sum_{i, j} k(r_i, g_j), over the rows
// i of strip a and every column j (the self terms count the pairs of the upper tiles, off-diagonal ones twice)
__global__ void __launch_bounds__(kKpdThreads)
kpd_strip_kernel(const double* __restrict__ g, int B, int d, int degree, double* __restrict__ partial) {
    extern __shared__ __align__(16) double kpd_smem[];
    __shared__ double red[kKpdThreads / 32];
    const int a = blockIdx.x, term = blockIdx.y, batch = blockIdx.z, nt = gridDim.x;
    const int ld = d | 1;   // odd row stride: the 16 column rows a warp reads fall in distinct banks
    double* xs = kpd_smem;
    double* ys = kpd_smem + kKpdTile * ld;
    const double* base = g + (long long)batch * 2 * B * d;
    const double* first = base + (term == 1 ? (long long)B * d : 0);
    const double* second = base + (term == 0 ? 0 : (long long)B * d);
    const double inv_d = 1.0 / d;
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;   // rows ty + 16u, columns tx + 16v of a tile
    kpd_load(first, a * kKpdTile, B, d, ld, xs);
    double acc = 0.0;
    for (int b = term == 2 ? 0 : a; b < nt; ++b) {
        __syncthreads();
        kpd_load(second, b * kKpdTile, B, d, ld, ys);
        __syncthreads();
        double dot[4][4] = {};
        for (int c = 0; c < d; ++c) {
            double xv[4], yv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) xv[u] = xs[(ty + 16 * u) * ld + c];
#pragma unroll
            for (int v = 0; v < 4; ++v) yv[v] = ys[(tx + 16 * v) * ld + c];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) dot[u][v] = fma(xv[u], yv[v], dot[u][v]);
        }
        const double w = term == 2 || b == a ? 1.0 : 2.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = a * kKpdTile + ty + 16 * u;
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const int j = b * kKpdTile + tx + 16 * v;
                if (i >= B || j >= B || (term != 2 && i == j)) continue;
                const double k1 = dot[u][v] * inv_d + 1.0;
                double kv = k1;
                for (int p = 1; p < degree; ++p) kv *= k1;
                acc += w * kv;
            }
        }
    }
    const double s = kpd_block_sum(acc, red);
    if (threadIdx.x == 0) partial[((long long)batch * 3 + term) * nt + a] = s;
}

// one block per batch: out = (S_rr + S_gg) / (B (B - 1)) - 2 S_rg / B^2
__global__ void __launch_bounds__(kKpdFinalThreads)
kpd_final_kernel(const double* __restrict__ partial, int nt, int B, double* __restrict__ out) {
    __shared__ double red[kKpdFinalThreads / 32];
    const int batch = blockIdx.x, per = (nt + kKpdFinalThreads - 1) / kKpdFinalThreads;
    double S[3];
    for (int t = 0; t < 3; ++t) {
        const double* p = partial + ((long long)batch * 3 + t) * nt;
        double s = 0.0;
        for (int k = threadIdx.x * per, k1 = min(k + per, nt); k < k1; ++k) s += p[k];
        S[t] = kpd_block_sum(s, red);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double b = (double)B;
        out[batch] = (S[0] + S[1]) / (b * (b - 1.0)) - 2.0 * S[2] / (b * b);
    }
}

constexpr size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

size_t kpd_gathered_bytes(int batches, int B, int d) { return align256((size_t)batches * 2 * B * d * sizeof(double)); }

int kpd_strips(int B) { return (B + kKpdTile - 1) / kKpdTile; }

}  // namespace

int launch_sampled_moments(const float* x, long long ldx, int d, const float* scale, const int* idx, int draws, int rows, double* sum,
                           double* sumsq, cudaStream_t stream) {
    moments_kernel<<<draws, kMomThreads, 0, stream>>>(x, ldx, d, scale, idx, rows, sum, sumsq);
    return cuda_ok(cudaGetLastError(), "sampled_moments launch");
}

size_t kpd_mmd_workspace_bytes(int batches, int B, int d) {
    return kpd_gathered_bytes(batches, B, d) + align256((size_t)batches * 3 * kpd_strips(B) * sizeof(double));
}

int launch_kpd_mmd(const float* real, long long ldr, const float* gen, long long ldg, int d, const float* scale, const int* idx_real,
                   const int* idx_gen, int batches, int B, int degree, double* out, void* workspace, cudaStream_t stream) {
    double* g = static_cast<double*>(workspace);
    double* partial = reinterpret_cast<double*>(static_cast<char*>(workspace) + kpd_gathered_bytes(batches, B, d));
    const long long total = (long long)batches * 2 * B * d;
    const int gather_blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    kpd_gather_kernel<<<gather_blocks, 256, 0, stream>>>(real, ldr, gen, ldg, d, scale, idx_real, idx_gen, batches, B, g);
    const size_t smem = 2 * (size_t)kKpdTile * (d | 1) * sizeof(double);
    if (smem > 48 * 1024)
        if (int rc = cuda_ok(cudaFuncSetAttribute(kpd_strip_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "kpd smem"))
            return rc;
    const int nt = kpd_strips(B);
    kpd_strip_kernel<<<dim3(nt, 3, batches), kKpdThreads, smem, stream>>>(g, B, d, degree, partial);
    kpd_final_kernel<<<batches, kKpdFinalThreads, 0, stream>>>(partial, nt, B, out);
    return cuda_ok(cudaGetLastError(), "kpd_mmd launch");
}

}  // namespace mmb
