// efp.cu — energy flow polynomials of a generated batch, in two column sets of one kernel (efp_kernel<D4>):
//   D4 = false (mmb_energy_flow_polynomials): the d = 1 EFP and the five connected 4-vertex, 4-edge multigraphs that W1-EFP of
//     Kansal et al. (arXiv:2211.10295) uses;
//   D4 = true (mmb_energy_flow_polynomials_d4): every EFP of degree d <= 4, the 36 features JetNet scores FPD and KPD on.
// Definitions: include/mmbridge.h and DESIGN.md §4.6d / §4.6f; numpy restatements: tests/efp_oracle.py, tests/efp_d4_oracle.py.
//
// One 128-thread block per jet.  The used particles are compacted into shared memory in slot order.  theta_ik = dR_ik^beta is
// computed once (dR^2 in fp64) and stored in fp32 as the upper triangle of 32 x 32 blocks (row stride 33), so that N = 256 needs 36
// blocks (152 KB) instead of a full 256 KB square.  The hot term M = Theta diag(z) Theta is never stored: for every upper
// output tile (I <= K) the block forms M_ik in fp32 registers (4 x 2 per thread) and at once adds the four pair terms that
// need it or theta_ik: each term an fp32 product, every sum fp64.  Every thread walks the same tiles in the same order and the block sums have a fixed shape,
// so the result is bit-identical from call to call.
//
// The d <= 4 set shares every line of that walk.  It adds the row sums c, r (theta^3, theta^4) and u = Theta diag(z) s in one more
// O(n^2) pass, twelve more O(n) row terms, and two more fp64 accumulators (the triangle and the triangle with a doubled edge)
// in the tile epilogue.  The shared columns are computed by the same statements in the same order, so they are bit-identical to
// the JetNet set's.  The 15 disconnected graphs are products of the 20 connected sums, formed in fp64 and rounded once.
#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

namespace {

constexpr int kEfpThreads = 128;
constexpr int kEfpTile = 32;
constexpr int kEfpLd = kEfpTile + 1;              // padded row of a stored block
constexpr int kEfpBlock = kEfpTile * kEfpLd;      // floats per stored block
constexpr double kEfpPi = 3.141592653589793, kEfpTwoPi = 6.283185307179586;

__device__ __forceinline__ double efp_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// index of the stored block (A, B), A <= B, among the upper blocks of an nb x nb grid
__device__ __forceinline__ int efp_blk(int A, int B, int nb) { return A * nb - A * (A - 1) / 2 + (B - A); }

// theta_ij from the triangle of blocks, either order of the indices
__device__ __forceinline__ float efp_theta(const float* th, int i, int k, int nb) {
    int A = i >> 5, B = k >> 5, r = i & 31, c = k & 31;
    if (A > B) { const int t = A; A = B; B = t; const int u = r; r = c; c = u; }
    return th[efp_blk(A, B, nb) * kEfpBlock + r * kEfpLd + c];
}

// row j (j = J*32 + jj) of Theta restricted to the 32 columns of block X: element x at p[jj * sj + x * sx]
__device__ __forceinline__ const float* efp_panel(const float* th, int J, int X, int nb, int& sj, int& sx) {
    if (J <= X) { sj = kEfpLd; sx = 1; return th + efp_blk(J, X, nb) * kEfpBlock; }
    sj = 1; sx = kEfpLd;
    return th + efp_blk(X, J, nb) * kEfpBlock;
}

// The connected sums of the d <= 4 set beyond the MMB_EFP_OBS of the JetNet set (which keep their slots 0..5): twelve row terms,
// sums over i of z_i times a product of s, q, c, r, u; then the two tile terms.
enum { kR2Double, kR2Path, kR3Triple, kR3PathDouble, kR3Path, kR3Star, kR4Quadruple, kR4TripleSingle, kR4DoubleDouble, kR4Path,
       kR4Star, kR4Fork, kEfpRowTerms };
enum { kT3Triangle, kT4TriangleDouble, kEfpTileTerms };
constexpr int kEfpRow0 = MMB_EFP_OBS, kEfpTile0 = kEfpRow0 + kEfpRowTerms, kEfpD4Sums = kEfpTile0 + kEfpTileTerms;   // 20
static_assert(kEfpD4Sums == 20, "20 connected loopless multigraphs with 1 <= d <= 4 edges");

// column c of the d <= 4 set is the product of the connected sums kEfpD4Factors[c][0..3] (-1: none; none at all: efp0 = 1)
#define EFP_R(t) (kEfpRow0 + t)
#define EFP_T(t) (kEfpTile0 + t)
__constant__ signed char kEfpD4Factors[MMB_EFPD4_OBS][4] = {
    {-1, -1, -1, -1},                                   // efp0
    {MMB_EFP_1, -1, -1, -1},                            // d = 1
    {EFP_R(kR2Double), -1, -1, -1}, {EFP_R(kR2Path), -1, -1, -1}, {MMB_EFP_1, MMB_EFP_1, -1, -1},
    {EFP_R(kR3Triple), -1, -1, -1}, {EFP_R(kR3PathDouble), -1, -1, -1}, {EFP_T(kT3Triangle), -1, -1, -1},
    {EFP_R(kR3Path), -1, -1, -1}, {EFP_R(kR3Star), -1, -1, -1},
    {MMB_EFP_1, EFP_R(kR2Double), -1, -1}, {MMB_EFP_1, EFP_R(kR2Path), -1, -1}, {MMB_EFP_1, MMB_EFP_1, MMB_EFP_1, -1},
    {EFP_R(kR4Quadruple), -1, -1, -1}, {EFP_R(kR4TripleSingle), -1, -1, -1}, {EFP_R(kR4DoubleDouble), -1, -1, -1},
    {EFP_T(kT4TriangleDouble), -1, -1, -1}, {MMB_EFP_4_SQUARE, -1, -1, -1}, {MMB_EFP_4_PAW, -1, -1, -1},
    {MMB_EFP_4_PATH_MID2, -1, -1, -1}, {MMB_EFP_4_PATH_END2, -1, -1, -1}, {MMB_EFP_4_STAR2, -1, -1, -1},
    {EFP_R(kR4Path), -1, -1, -1}, {EFP_R(kR4Star), -1, -1, -1}, {EFP_R(kR4Fork), -1, -1, -1},
    {MMB_EFP_1, EFP_R(kR3Triple), -1, -1}, {MMB_EFP_1, EFP_R(kR3PathDouble), -1, -1}, {MMB_EFP_1, EFP_T(kT3Triangle), -1, -1},
    {MMB_EFP_1, EFP_R(kR3Path), -1, -1}, {MMB_EFP_1, EFP_R(kR3Star), -1, -1},
    {EFP_R(kR2Double), EFP_R(kR2Double), -1, -1}, {EFP_R(kR2Double), EFP_R(kR2Path), -1, -1},
    {EFP_R(kR2Path), EFP_R(kR2Path), -1, -1}, {MMB_EFP_1, MMB_EFP_1, EFP_R(kR2Double), -1},
    {MMB_EFP_1, MMB_EFP_1, EFP_R(kR2Path), -1}, {MMB_EFP_1, MMB_EFP_1, MMB_EFP_1, MMB_EFP_1}};
#undef EFP_R
#undef EFP_T

template <bool D4> struct EfpSet {   // sums reduced per block, columns written per jet
    static constexpr int kSums = D4 ? kEfpD4Sums : MMB_EFP_OBS, kOut = D4 ? (int)MMB_EFPD4_OBS : (int)MMB_EFP_OBS;
};

}  // namespace

template <bool D4>
__global__ void __launch_bounds__(kEfpThreads, 4)   // min blocks: without it ptxas trims registers and spills around the calls
efp_kernel(const float* __restrict__ x, const uint8_t* __restrict__ mask, float3 mean, float3 sd, int N, int nb_max, double beta,
           float* __restrict__ out) {
    using Set = EfpSet<D4>;
    extern __shared__ __align__(16) unsigned char efp_smem[];
    __shared__ double red[kEfpThreads / 32][Set::kSums];
    __shared__ double s_ptsum;
    __shared__ int s_n;
    const int P = nb_max * kEfpTile;
    double* s = reinterpret_cast<double*>(efp_smem);   // s_i = sum_j z_j theta_ij
    double* q = s + P;                                 // q_i = sum_j z_j theta_ij^2
    double* c3 = q + P;                                // d <= 4 only: c_i = sum_j z_j theta_ij^3, r_i (^4), u_i = sum_k theta_ik z_k s_k
    double* r4 = c3 + P;
    double* u = r4 + P;
    float* z = reinterpret_cast<float*>(D4 ? u + P : q + P);   // pt, then z
    float* eta = z + P;
    float* phi = eta + P;
    float* th = phi + P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, jet = blockIdx.x;
    float* o = out + (size_t)jet * Set::kOut;

    // inputs: (x * std + mean) in fp32; used iff mask != 0 && pt > 0; compacted in slot order by warp 0, pt summed in fp64
    if (warp == 0) {
        int base = 0;
        double ptsum = 0.0;
        for (int n0 = 0; n0 < N; n0 += 32) {
            const int slot = n0 + lane;
            const size_t p = (size_t)jet * N + slot;
            float c0 = 0.0f, c1 = 0.0f, c2 = 0.0f;
            bool used = false;
            if (slot < N && mask[p]) {
                c0 = __fadd_rn(__fmul_rn(x[p * 3], sd.x), mean.x);
                c1 = __fadd_rn(__fmul_rn(x[p * 3 + 1], sd.y), mean.y);
                c2 = __fadd_rn(__fmul_rn(x[p * 3 + 2], sd.z), mean.z);
                used = c0 > 0.0f;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, used);
            if (used) {
                const int i = base + __popc(bal & ((1u << lane) - 1u));
                z[i] = c0; eta[i] = c1; phi[i] = c2;
                ptsum += c0;
            }
            base += __popc(bal);
        }
        ptsum = efp_warp_sum(ptsum);
        if (lane == 0) { s_n = base; s_ptsum = ptsum; }
    }
    __syncthreads();
    const int n = s_n;
    if (n == 0) {   // no used particle: z is undefined
        if (threadIdx.x < Set::kOut) o[threadIdx.x] = __int_as_float(0x7fffffff);
        return;
    }
    const int nb = (n + kEfpTile - 1) / kEfpTile, np = nb * kEfpTile;
    const double ptsum = s_ptsum;
    for (int i = threadIdx.x; i < np; i += kEfpThreads) z[i] = i < n ? (float)((double)z[i] / ptsum) : 0.0f;

    // theta in the upper blocks: fp64 dR (dphi wrapped into [-pi, pi]) to the power beta, 0 on the diagonal and in the padding
    const int stored = nb * (nb + 1) / 2 * kEfpTile * kEfpTile;
    for (int e = threadIdx.x; e < stored; e += kEfpThreads) {
        const int b = e >> 10, r = (e >> 5) & 31, c = e & 31;
        int A = 0, rem = b;
        while (rem >= nb - A) { rem -= nb - A; ++A; }
        const int i = A * kEfpTile + r, k = (A + rem) * kEfpTile + c;
        float t = 0.0f;
        if (i < n && k < n && i != k) {
            const double deta = (double)eta[i] - (double)eta[k];
            double dphi = (double)phi[i] - (double)phi[k];
            if (dphi > kEfpPi) dphi -= kEfpTwoPi;
            else if (dphi < -kEfpPi) dphi += kEfpTwoPi;
            const double dr2 = deta * deta + dphi * dphi;
            const float r2 = (float)dr2;   // theta is stored in fp32: the root or power of the rounded dR^2 adds an ulp or two
            t = beta == 1.0 ? sqrtf(r2) : (r2 > 0.0f ? powf(r2, (float)(0.5 * beta)) : 0.0f);
        }
        th[b * kEfpBlock + r * kEfpLd + c] = t;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < np; i += kEfpThreads) {
        double si = 0.0, qi = 0.0;
        for (int k = 0; k < n; ++k) {
            const double t = efp_theta(th, i, k, nb), zk = z[k];
            si += zk * t;
            qi += zk * t * t;
        }
        s[i] = si;
        q[i] = qi;
    }
    __syncthreads();
    if constexpr (D4) {   // a pass of its own, so that s and q come from the same instructions in both sets
        for (int i = threadIdx.x; i < np; i += kEfpThreads) {
            double ci = 0.0, ri = 0.0, ui = 0.0;
            for (int k = 0; k < n; ++k) {
                const double t = efp_theta(th, i, k, nb), zk = z[k], t2 = t * t;
                ci += zk * t2 * t;
                ri += zk * t2 * t2;
                ui += t * zk * s[k];
            }
            c3[i] = ci;
            r4[i] = ri;
            u[i] = ui;
        }
        __syncthreads();
    }

    // acc: efp1, square, paw, path_mid2, path_end2, star2 (per-thread fp64 partials)
    double acc[MMB_EFP_OBS] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n; i += kEfpThreads) {
        const double zi = z[i], si = s[i];
        acc[MMB_EFP_1] += zi * si;
        acc[MMB_EFP_4_STAR2] += zi * q[i] * si * si;
    }
    if constexpr (D4) {   // the twelve row terms, reduced per warp now so that they are not live through the tile walk
        double e[kEfpRowTerms] = {};
        for (int i = threadIdx.x; i < n; i += kEfpThreads) {
            const double zi = z[i], si = s[i], qi = q[i], ci = c3[i], ri = r4[i], ui = u[i], zs = zi * si, zss = zs * si;
            e[kR2Double] += zi * qi;
            e[kR2Path] += zss;
            e[kR3Triple] += zi * ci;
            e[kR3PathDouble] += zi * qi * si;
            e[kR3Path] += zs * ui;
            e[kR3Star] += zss * si;
            e[kR4Quadruple] += zi * ri;
            e[kR4TripleSingle] += zi * ci * si;
            e[kR4DoubleDouble] += zi * qi * qi;
            e[kR4Path] += zi * ui * ui;
            e[kR4Star] += zss * si * si;
            e[kR4Fork] += zss * ui;
        }
#pragma unroll
        for (int g = 0; g < kEfpRowTerms; ++g) {
            const double v = efp_warp_sum(e[g]);
            if (lane == 0) red[warp][kEfpRow0 + g] = v;
        }
    }
    double tri[kEfpTileTerms] = {0.0, 0.0};   // d <= 4 only: the triangle and the triangle with a doubled edge
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;   // rows ty*4 .. +3, columns tx*2 .. +1 of a 32 x 32 tile
    for (int I = 0; I < nb; ++I) {
        for (int K = I; K < nb; ++K) {
            float m[4][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}, {0.0f, 0.0f}, {0.0f, 0.0f}};
            for (int J = 0; J < nb; ++J) {
                int sji = 0, sxi = 0, sjk = 0, sxk = 0;
                const float* pi = efp_panel(th, J, I, nb, sji, sxi) + ty * 4 * sxi;
                const float* pk = efp_panel(th, J, K, nb, sjk, sxk) + tx * 2 * sxk;
                const float* zj = z + J * kEfpTile;
#pragma unroll 4
                for (int jj = 0; jj < kEfpTile; ++jj) {
                    const float w = zj[jj];
                    float a[4], c[2];
#pragma unroll
                    for (int u = 0; u < 4; ++u) a[u] = pi[jj * sji + u * sxi] * w;
#pragma unroll
                    for (int v = 0; v < 2; ++v) c[v] = pk[jj * sjk + v * sxk];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int v = 0; v < 2; ++v) m[u][v] = fmaf(a[u], c[v], m[u][v]);
                }
            }
            // the ordered pairs (i, k) of this tile; an off-diagonal tile also stands for (k, i)
            const float* tik = th + efp_blk(I, K, nb) * kEfpBlock;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int r = ty * 4 + u, i = I * kEfpTile + r;
                const float zi = z[i], si = (float)s[i], qi = (float)q[i];
#pragma unroll
                for (int v = 0; v < 2; ++v) {   // each term a product of a few fp32 factors, the sums fp64
                    const int c = tx * 2 + v, k = K * kEfpTile + c;
                    const float zz = zi * z[k], sk = (float)s[k], qk = (float)q[k], t = tik[r * kEfpLd + c], M = m[u][v];
                    if (I == K) {
                        acc[MMB_EFP_4_SQUARE] += (double)(zz * M * M);
                        acc[MMB_EFP_4_PAW] += (double)(zz * t * M * si);
                        acc[MMB_EFP_4_PATH_MID2] += (double)(zz * si * sk * t * t);
                        acc[MMB_EFP_4_PATH_END2] += (double)(zz * qi * t * sk);
                        if constexpr (D4) {
                            tri[kT3Triangle] += (double)(zz * t * M);
                            tri[kT4TriangleDouble] += (double)(zz * t * t * M);
                        }
                    } else {
                        acc[MMB_EFP_4_SQUARE] += (double)(2.0f * zz * M * M);
                        acc[MMB_EFP_4_PAW] += (double)(zz * t * M * (si + sk));
                        acc[MMB_EFP_4_PATH_MID2] += (double)(2.0f * zz * si * sk * t * t);
                        acc[MMB_EFP_4_PATH_END2] += (double)(zz * t * (qi * sk + qk * si));
                        if constexpr (D4) {
                            tri[kT3Triangle] += (double)(2.0f * zz * t * M);
                            tri[kT4TriangleDouble] += (double)(2.0f * zz * t * t * M);
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int g = 0; g < MMB_EFP_OBS; ++g) {
        const double v = efp_warp_sum(acc[g]);
        if (lane == 0) red[warp][g] = v;
    }
    if constexpr (D4) {
#pragma unroll
        for (int g = 0; g < kEfpTileTerms; ++g) {
            const double v = efp_warp_sum(tri[g]);
            if (lane == 0) red[warp][kEfpTile0 + g] = v;
        }
    }
    __syncthreads();
    if constexpr (!D4) {
        if (threadIdx.x < MMB_EFP_OBS) {
            double v = 0.0;
            for (int w = 0; w < kEfpThreads / 32; ++w) v += red[w][threadIdx.x];
            o[threadIdx.x] = (float)v;
        }
    } else {   // the 20 connected sums (added over the warps as above), then every column as a product of them, rounded once
        __shared__ double sum[kEfpD4Sums];
        if (threadIdx.x < kEfpD4Sums) {
            double v = 0.0;
            for (int w = 0; w < kEfpThreads / 32; ++w) v += red[w][threadIdx.x];
            sum[threadIdx.x] = v;
        }
        __syncthreads();
        if (threadIdx.x < MMB_EFPD4_OBS) {
            double v = 1.0;
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                const int g = kEfpD4Factors[threadIdx.x][f];
                if (g >= 0) v *= sum[g];
            }
            o[threadIdx.x] = (float)v;
        }
    }
}

// s, q (and for d <= 4 c, r, u) in fp64, z, eta, phi in fp32 per padded particle, then the upper triangle of Theta blocks;
// N = 256: 152 KB + 7 KB, with the d <= 4 row sums + 6 KB
static size_t efp_smem_bytes(int nb, bool d4) {
    const size_t P = (size_t)nb * kEfpTile;
    return P * ((d4 ? 5 : 2) * sizeof(double) + 3 * sizeof(float)) + (size_t)nb * (nb + 1) / 2 * kEfpBlock * sizeof(float);
}

template <bool D4>
static int launch_efp(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float beta, float* out,
                      cudaStream_t stream, const char* what) {
    const float3 m = mean ? make_float3(mean[0], mean[1], mean[2]) : make_float3(0.0f, 0.0f, 0.0f);
    const float3 s = sd ? make_float3(sd[0], sd[1], sd[2]) : make_float3(1.0f, 1.0f, 1.0f);
    const int nb = N > 0 ? (N + kEfpTile - 1) / kEfpTile : 1;
    const size_t smem = efp_smem_bytes(nb, D4);
    // the opt-in above 48 KB covers static + dynamic shared memory: the d <= 4 set's 816 static bytes push N = 128 (48 896 B
    // dynamic) over the default limit
    cudaFuncAttributes fa{};
    if (int rc = cuda_ok(cudaFuncGetAttributes(&fa, efp_kernel<D4>), "efp attributes")) return rc;
    if (fa.sharedSizeBytes + smem > 48 * 1024)
        if (int rc = cuda_ok(cudaFuncSetAttribute(efp_kernel<D4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "efp smem"))
            return rc;
    efp_kernel<D4><<<B, kEfpThreads, smem, stream>>>(x, mask, m, s, N, nb, (double)beta, out);
    return cuda_ok(cudaGetLastError(), what);
}

int launch_energy_flow_polynomials(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float beta,
                                   float* out, cudaStream_t stream) {
    return launch_efp<false>(x, mask, mean, sd, B, N, beta, out, stream, "energy_flow_polynomials launch");
}

int launch_energy_flow_polynomials_d4(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N,
                                      float beta, float* out, cudaStream_t stream) {
    return launch_efp<true>(x, mask, mean, sd, B, N, beta, out, stream, "energy_flow_polynomials_d4 launch");
}

}  // namespace mmb
