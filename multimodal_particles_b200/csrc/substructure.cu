// substructure.cu — jet substructure of a generated batch: N-subjettiness tau1..tau3 on exclusive kt / WTA_pt axes and the
// energy correlation functions e2, e3, D2 (JetClassHighLevelFeatures.substructure, mp/data/particle_clouds/jets.py:204-240).
// Definitions: include/mmbridge.h and DESIGN.md §4.6; CPU restatement: oracle_substructure/mmbo_substructure.c.
//
// One 128-thread block per jet.  The used particles are compacted into shared memory in fp64.  Warp 0 runs the clustering
// with nearest-neighbour bookkeeping (FastJet's NNH idea): every object keeps its best candidate, a step is a warp argmin
// over those, and only the objects whose candidate took part in the step are rescanned; the others compare their distance
// to the merged object.  Every distance is spelled with __dmul_rn / __dadd_rn in the oracle's order, so the merge
// sequence and the axes are bit-identical to it.  Meanwhile warps 1..3 (and warp 0 once it is done) sum e3 over a triangle
// of dR^beta in fp32, one row per warp at a time, rows handed out by a shared counter; row sums land in shared memory and
// are added in row order, so the result does not depend on which warp took which row.
#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

namespace {

constexpr int kSubWarps = 4;
constexpr double kPi = 3.141592653589793, kTwoPi = 6.283185307179586;

__device__ __forceinline__ double delta_r2(double eta_a, double phi_a, double eta_b, double phi_b) {
    const double deta = __dsub_rn(eta_a, eta_b);
    double dphi = __dsub_rn(phi_a, phi_b);
    if (dphi > kPi) dphi = __dsub_rn(dphi, kTwoPi);
    else if (dphi < -kPi) dphi = __dadd_rn(dphi, kTwoPi);
    return __dadd_rn(__dmul_rn(deta, deta), __dmul_rn(dphi, dphi));
}

// dR^beta from dR^2, within a few ulp of the oracle's sqrt / pow; rsqrt and exp / log are inline, where sqrt and pow would call
// out-of-line slow paths from inside the loops and cost the kernel body its registers
__device__ __forceinline__ double angle_pow(double dr2, double beta) {
    if (beta == 1.0) return dr2 > 0.0 ? dr2 * rsqrt(dr2) : 0.0;
    return exp(0.5 * beta * log(dr2));
}

// (d, code) order of the tie rule; code = lower * 512 + upper, a beam candidate of i being i * 512 + i
__device__ __forceinline__ bool key_less(double d, int c, double d2, int c2) { return d < d2 || (d == d2 && c < c2); }

__device__ __forceinline__ void warp_argmin(double& d, int& c) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, d, o);
        const int oc = __shfl_xor_sync(0xffffffffu, c, o);
        if (key_less(od, oc, d, c)) { d = od; c = oc; }
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct SubShared {
    double *pt, *eta, *phi, *z;    // used particles, compacted in slot order
    double *opt, *nnd, *e3row;     // current pt of each object, distance of its best candidate; e3 row sums
    int *slot, *dir, *nnc;         // slot of each particle; particle whose direction an object carries; code of its best candidate
    unsigned char* alive;
    float* ang;                    // dR^beta of the pair (i, k), k > i, at tri(i) + k - i - 1
};

__device__ __forceinline__ int tri(int i, int n) { return i * (2 * n - i - 1) / 2; }

// d_ij of two present objects (the oracle's order of operations: lower index first)
__device__ __forceinline__ double pair_d(const SubShared s, int i, int j, double invR2, int& code) {
    const int lo = i < j ? i : j, hi = i < j ? j : i;
    const double p2l = __dmul_rn(s.opt[lo], s.opt[lo]), p2h = __dmul_rn(s.opt[hi], s.opt[hi]);
    const double m = p2l < p2h ? p2l : p2h;
    const int a = s.dir[lo], b = s.dir[hi];
    code = lo * 512 + hi;
    return __dmul_rn(__dmul_rn(m, delta_r2(s.eta[a], s.phi[a], s.eta[b], s.phi[b])), invR2);
}

// best candidate of object k over the beam and every other present object, the warp's lanes splitting the partners
__device__ __forceinline__ void rescan(const SubShared s, int k, int n, double invR2, int lane) {
    double bd = INFINITY;
    int bc = 0x7fffffff;
    for (int j = lane; j < n; j += 32) {
        if (!s.alive[j]) continue;
        double d;
        int c;
        if (j == k) { d = __dmul_rn(s.opt[k], s.opt[k]); c = k * 512 + k; }
        else d = pair_d(s, k, j, invR2, c);
        if (key_less(d, c, bd, bc)) { bd = d; bc = c; }
    }
    warp_argmin(bd, bc);
    if (lane == 0) { s.nnd[k] = bd; s.nnc[k] = bc; }
    __syncwarp();
}

// the present objects' directions, in ascending object index, as indices of used particles
__device__ __forceinline__ void record_axes(const SubShared s, int n, int* dst, int lane) {
    int base = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        const bool on = i < n && s.alive[i];
        const unsigned bal = __ballot_sync(0xffffffffu, on);
        if (on) dst[base + __popc(bal & ((1u << lane) - 1u))] = s.dir[i];
        base += __popc(bal);
    }
}

// exclusive kt clustering with WTA_pt recombination down to one object (warp 0)
__device__ __forceinline__ void cluster(const SubShared s, int n, double invR2, int* ax, int lane) {
    int left = n;
    for (;;) {
        if (left <= 3) record_axes(s, n, ax + (left == 1 ? 0 : left == 2 ? 1 : 3), lane);
        if (left == 1) break;
        double bd = INFINITY;
        int bc = 0x7fffffff;
        for (int i = lane; i < n; i += 32)
            if (s.alive[i] && key_less(s.nnd[i], s.nnc[i], bd, bc)) { bd = s.nnd[i]; bc = s.nnc[i]; }
        warp_argmin(bd, bc);
        const int lo = bc >> 9, hi = bc & 511;
        const bool merge = lo != hi;
        if (lane == 0) {
            if (merge) {   // into the lower index, direction of the harder object (the lower index on a pt tie)
                if (s.opt[hi] > s.opt[lo]) s.dir[lo] = s.dir[hi];
                s.opt[lo] = __dadd_rn(s.opt[lo], s.opt[hi]);
                s.alive[hi] = 0;
            } else {
                s.alive[lo] = 0;   // beam step
            }
        }
        __syncwarp();
        --left;
        // bookkeeping: objects whose candidate involved lo or hi (and the merged object itself) rescan; the others only
        // compare their distance to the merged object
        for (int i0 = 0; i0 < n; i0 += 32) {
            const int k = i0 + lane;
            bool again = false;
            if (k < n && s.alive[k]) {
                const int c = s.nnc[k], partner = (c >> 9) == k ? (c & 511) : (c >> 9);
                again = (merge && k == lo) || partner == lo || partner == hi;
                if (!again && merge) {
                    int code;
                    const double d = pair_d(s, k, lo, invR2, code);
                    if (key_less(d, code, s.nnd[k], c)) { s.nnd[k] = d; s.nnc[k] = code; }
                }
            }
            unsigned todo = __ballot_sync(0xffffffffu, again);
            __syncwarp();
            while (todo) {
                const int b = __ffs(todo) - 1;
                todo &= todo - 1;
                rescan(s, i0 + b, n, invR2, lane);
            }
        }
    }
}

// the ratios of one jet's row; out of line so that the slow paths of the divisions need no registers of the kernel body
__device__ __noinline__ void write_row(float* o, double t1, double t2, double t3, double d0, double e2, double e3) {
    t1 /= d0; t2 /= d0; t3 /= d0;
    o[MMB_SUB_TAU1] = (float)t1; o[MMB_SUB_TAU2] = (float)t2; o[MMB_SUB_TAU3] = (float)t3;
    o[MMB_SUB_TAU21] = (float)(t2 / t1); o[MMB_SUB_TAU32] = (float)(t3 / t2);
    o[MMB_SUB_E2] = (float)e2; o[MMB_SUB_E3] = (float)e3; o[MMB_SUB_D2] = (float)(e3 / (e2 * e2 * e2));
}

}  // namespace

__global__ void __launch_bounds__(kSubWarps * 32, 4)   // min blocks: without it ptxas trims registers and spills around the calls
jet_substructure_kernel(const float* __restrict__ x, const uint8_t* __restrict__ mask, float3 mean, float3 sd, int N, double invR2,
                        double beta, double d0_per_pt, float* __restrict__ out, int16_t* __restrict__ axes) {
    extern __shared__ __align__(16) unsigned char sub_smem[];
    __shared__ double red[kSubWarps][4], s_ptsum;
    __shared__ int s_n, s_row, s_ax[6];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, jet = blockIdx.x;
    SubShared s;
    {
        double* d = reinterpret_cast<double*>(sub_smem);
        s.pt = d; s.eta = d + N; s.phi = d + 2 * N; s.z = d + 3 * N; s.opt = d + 4 * N; s.nnd = d + 5 * N; s.e3row = d + 6 * N;
        int* q = reinterpret_cast<int*>(d + 7 * N);
        s.slot = q; s.dir = q + N; s.nnc = q + 2 * N;
        s.ang = reinterpret_cast<float*>(q + 3 * N);
        s.alive = reinterpret_cast<unsigned char*>(s.ang + (size_t)N * (N - 1) / 2);
    }

    // inputs: (x * std + mean) in fp32; used iff mask != 0 && pt > 0; compacted in slot order by warp 0
    if (warp == 0) {
        int base = 0;
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
                s.pt[i] = c0; s.eta[i] = c1; s.phi[i] = c2; s.slot[i] = slot;
                s.opt[i] = c0; s.dir[i] = i; s.alive[i] = 1;
            }
            base += __popc(bal);
        }
        if (lane == 0) { s_n = base; s_row = 0; }
    }
    __syncthreads();
    const int n = s_n;
    float* o = out + (size_t)jet * MMB_SUB_OBS;
    if (n < 3) {   // undefined: NaN, axes -1
        if (threadIdx.x < MMB_SUB_OBS) o[threadIdx.x] = __int_as_float(0x7fffffff);
        if (axes && threadIdx.x < 6) axes[(size_t)jet * 6 + threadIdx.x] = -1;
        return;
    }

    // scalar pt sum (fixed order: every warp sums the same way), z_i; then, one row per warp at a time: the dR^beta triangle,
    // e2 and the first candidate of every object
    double ptsum = 0.0;
    for (int i = lane; i < n; i += 32) ptsum += s.pt[i];
    ptsum = warp_sum(ptsum);
    for (int i = threadIdx.x; i < n; i += blockDim.x) s.z[i] = s.pt[i] / ptsum;
    __syncthreads();
    double e2 = 0.0;
    for (int i = warp; i < n; i += kSubWarps) {
        const int t0 = tri(i, n) - i - 1;
        for (int k = i + 1 + lane; k < n; k += 32) {
            const double a = angle_pow(delta_r2(s.eta[i], s.phi[i], s.eta[k], s.phi[k]), beta);
            s.ang[t0 + k] = (float)a;
            e2 += s.z[i] * s.z[k] * a;
        }
        rescan(s, i, n, invR2, lane);
    }
    e2 = warp_sum(e2);
    if (lane == 0) red[warp][3] = e2;   // parked in shared memory: nothing fp64 stays live across the phases below
    if (threadIdx.x == 0) s_ptsum = ptsum;
    __syncthreads();

    // warp 0 clusters; every warp takes e3 rows from the shared counter (warp 0 once the clustering is done)
    if (warp == 0) cluster(s, n, invR2, s_ax, lane);
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(&s_row, 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= n - 2) break;
        const float* Ai = s.ang + tri(i, n) - i - 1;
        double acc = 0.0;
        for (int j = i + 1; j < n - 1; ++j) {
            const float* Aj = s.ang + tri(j, n) - j - 1;
            double inner = 0.0;
            for (int k = j + 1 + lane; k < n; k += 32) inner += s.z[k] * (double)(Ai[k] * Aj[k]);
            acc += s.z[j] * (double)Ai[j] * inner;
        }
        acc = warp_sum(acc);
        if (lane == 0) s.e3row[i] = s.z[i] * acc;
    }
    __syncthreads();

    // N-subjettiness on the three axis sets
    const int a0 = s_ax[0], a1 = s_ax[1], a2 = s_ax[2], a3 = s_ax[3], a4 = s_ax[4], a5 = s_ax[5];
    double t1 = 0.0, t2 = 0.0, t3 = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double e = s.eta[i], f = s.phi[i], p = s.pt[i];
        const double d0 = delta_r2(e, f, s.eta[a0], s.phi[a0]);
        const double d1 = delta_r2(e, f, s.eta[a1], s.phi[a1]), d2 = delta_r2(e, f, s.eta[a2], s.phi[a2]);
        const double d3 = delta_r2(e, f, s.eta[a3], s.phi[a3]), d4 = delta_r2(e, f, s.eta[a4], s.phi[a4]);
        const double d5 = delta_r2(e, f, s.eta[a5], s.phi[a5]);
        const double m2 = d1 < d2 ? d1 : d2, m34 = d3 < d4 ? d3 : d4, m3 = m34 < d5 ? m34 : d5;
        t1 += p * angle_pow(d0, beta);
        t2 += p * angle_pow(m2, beta);
        t3 += p * angle_pow(m3, beta);
    }
    t1 = warp_sum(t1); t2 = warp_sum(t2); t3 = warp_sum(t3);
    if (lane == 0) { red[warp][0] = t1; red[warp][1] = t2; red[warp][2] = t3; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tau[3] = {0.0, 0.0, 0.0}, e2s = 0.0, e3 = 0.0;
        for (int w = 0; w < kSubWarps; ++w) {
            for (int t = 0; t < 3; ++t) tau[t] += red[w][t];
            e2s += red[w][3];
        }
        for (int i = 0; i < n - 2; ++i) e3 += s.e3row[i];
        write_row(o, tau[0], tau[1], tau[2], s_ptsum * d0_per_pt, e2s, e3);
    }
    if (axes && threadIdx.x < 6) axes[(size_t)jet * 6 + threadIdx.x] = (int16_t)s.slot[s_ax[threadIdx.x]];
}

static size_t substructure_smem_bytes(int N) {
    return (size_t)N * (7 * sizeof(double) + 3 * sizeof(int)) + (size_t)N * (N - 1) / 2 * sizeof(float) + (size_t)N;
}

int launch_jet_substructure(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float R, float beta,
                            float* out, int16_t* axes, cudaStream_t stream) {
    const float3 m = mean ? make_float3(mean[0], mean[1], mean[2]) : make_float3(0.0f, 0.0f, 0.0f);
    const float3 s = sd ? make_float3(sd[0], sd[1], sd[2]) : make_float3(1.0f, 1.0f, 1.0f);
    const size_t smem = substructure_smem_bytes(N);
    if (smem > 48 * 1024)
        if (int rc = cuda_ok(cudaFuncSetAttribute(jet_substructure_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                             "substructure smem"))
            return rc;
    // 1 / R^2 and R^beta in host fp64, the same operations as the oracle
    const double R2 = (double)R * (double)R, invR2 = 1.0 / R2, b = (double)beta, Rb = b == 1.0 ? sqrt(R2) : pow(R2, 0.5 * b);
    jet_substructure_kernel<<<B, kSubWarps * 32, smem, stream>>>(x, mask, m, s, N, invR2, b, Rb, out, axes);
    return cuda_ok(cudaGetLastError(), "jet_substructure launch");
}

}  // namespace mmb
