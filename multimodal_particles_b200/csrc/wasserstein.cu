// wasserstein.cu — exact 1-D Wasserstein distance (W1) between two samples, per column, on the device
// (JetClassHighLevelFeatures.Wassertein1D, mp/data/particle_clouds/jets.py:329-332, which calls scipy.stats.wasserstein_distance).
// Definition: include/mmbridge.h and DESIGN.md §4.6c.
//
// Three stream-ordered stages, all in the caller's workspace:
//   1. w1_keys_kernel copies every column out of the caller's strided rows into order-preserving uint32 keys (non-finite
//      values become one canonical key that sorts after every finite value, -0 becomes +0) and counts the finite values.
//   2. One cub::DeviceRadixSort per column and sample (keys only: the result is a function of the multiset of values).
//   3. w1_merge_kernel walks the merged sequence of the two sorted columns in tiles of kW1Tile terms; a thread finds its
//      start on the merge path by binary search and walks kW1Items terms, a block adds its threads' sums in a fixed tree and
//      writes one fp64 partial.  w1_final_kernel adds the partials of each column in a fixed order and divides by n' m'.
// The tile is a compile-time constant, so the result depends only on the sorted samples: it is bit-identical from call to call
// and for any order of the rows.
#include <cub/device/device_radix_sort.cuh>

#include "mmb_internal.h"

namespace mmb {

namespace {

constexpr int kW1Threads = 256;
constexpr int kW1Items = 16;
constexpr long long kW1Tile = (long long)kW1Threads * kW1Items;
constexpr uint32_t kNoKey = 0xFFFFFFFFu;   // non-finite values; also the sentinel past the end of a sample
constexpr int kKeyBlocks = 4096;

__device__ __forceinline__ uint32_t w1_key(float v) {
    if (!isfinite(v)) return kNoKey;
    const uint32_t b = __float_as_uint(v == 0.0f ? 0.0f : v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);   // unsigned order of the keys = order of the values
}

__device__ __forceinline__ double w1_value(uint32_t k) {
    return (double)__uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// rows [rows][ld] f32 -> keys [K][rows]; finite[c] += number of finite values of column c
__global__ void __launch_bounds__(kW1Threads) w1_keys_kernel(const float* __restrict__ v, long long ld, long long rows, int K,
                                                             uint32_t* __restrict__ keys, unsigned long long* __restrict__ finite) {
    __shared__ unsigned int cnt[MMB_W1_MAX_K];
    for (int c = threadIdx.x; c < K; c += blockDim.x) cnt[c] = 0;
    __syncthreads();
    const long long total = rows * K;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / K;
        const int c = (int)(e - r * K);
        const uint32_t key = w1_key(v[r * ld + c]);
        keys[c * rows + r] = key;
        if (key != kNoKey) atomicAdd(&cnt[c], 1u);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < K; c += blockDim.x)
        if (cnt[c]) atomicAdd(&finite[c], (unsigned long long)cnt[c]);
}

// number of a-elements among the first d elements of the merge of a[0..na) and b[0..nb), a first on ties
__device__ __forceinline__ long long merge_split(const uint32_t* __restrict__ a, long long na, const uint32_t* __restrict__ b,
                                                 long long nb, long long d) {
    long long lo = d > nb ? d - nb : 0, hi = d < na ? d : na;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (a[mid] <= b[d - 1 - mid]) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ double block_sum(double s, double* red) {
    red[threadIdx.x] = s;
    __syncthreads();
    for (int h = kW1Threads / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

// grid (tiles, K): partial[c][tile] = sum over the terms k of the tile of |i_k m' - j_k n'| (z_{k+1} - z_k), k < n' + m' - 1
__global__ void __launch_bounds__(kW1Threads) w1_merge_kernel(const uint32_t* __restrict__ xs, long long n, const uint32_t* __restrict__ ys,
                                                              long long m, const unsigned long long* __restrict__ finite, int K,
                                                              double* __restrict__ partial) {
    __shared__ double red[kW1Threads];
    const int c = blockIdx.y;
    const long long nx = (long long)finite[c], ny = (long long)finite[K + c];
    const uint32_t* a = xs + c * n;
    const uint32_t* b = ys + c * m;
    const long long terms = nx + ny - 1;
    const long long k0 = blockIdx.x * kW1Tile + (long long)threadIdx.x * kW1Items;
    double s = 0.0;
    if (nx > 0 && ny > 0 && k0 < terms) {
        long long i = merge_split(a, nx, b, ny, k0), j = k0 - i;
        uint32_t va = i < nx ? a[i] : kNoKey, vb = j < ny ? b[j] : kNoKey;
        uint32_t cur = min(va, vb);
        const long long k1 = min(k0 + kW1Items, terms);
        for (long long k = k0; k < k1; ++k) {   // take z_k; then i + j = k + 1 values are <= z_k
            if (va <= vb) {
                ++i;
                va = i < nx ? a[i] : kNoKey;
            } else {
                ++j;
                vb = j < ny ? b[j] : kNoKey;
            }
            const uint32_t nxt = min(va, vb);
            if (nxt != cur) {   // equal values (ties within or across the samples) contribute nothing
                const long long w = i * ny - j * nx;   // exact: |w| <= 2^62
                s += (double)(w < 0 ? -w : w) * (w1_value(nxt) - w1_value(cur));
            }
            cur = nxt;
        }
    }
    const double t = block_sum(s, red);
    if (threadIdx.x == 0) partial[c * (long long)gridDim.x + blockIdx.x] = t;
}

// one block: out[c] = sum of the partials of column c / (n' m'), NaN when a sample has no finite value
__global__ void __launch_bounds__(kW1Threads) w1_final_kernel(const double* __restrict__ partial, int tiles,
                                                              const unsigned long long* __restrict__ finite, int K,
                                                              double* __restrict__ out, long long* __restrict__ n_used) {
    __shared__ double red[kW1Threads];
    const int per = (tiles + kW1Threads - 1) / kW1Threads;
    for (int c = 0; c < K; ++c) {
        const double* p = partial + (long long)c * tiles;
        double s = 0.0;
        for (int t = threadIdx.x * per, t1 = min(t + per, tiles); t < t1; ++t) s += p[t];
        const double total = block_sum(s, red);
        if (threadIdx.x == 0) {
            const unsigned long long nx = finite[c], ny = finite[K + c];
            out[c] = (nx && ny) ? total / ((double)nx * (double)ny) : __longlong_as_double(0x7FF8000000000000LL);
            if (n_used) {
                n_used[c] = (long long)nx;
                n_used[K + c] = (long long)ny;
            }
        }
    }
}

constexpr size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct W1Layout {
    size_t counts, keys_a, keys_b, partial, temp, temp_bytes, total;
    int tiles;
};

// workspace: finite counts [2K] u64 | keys [K(n+m)] u32 | alternate keys [K(n+m)] u32 | partials [K][tiles] f64 | CUB temp
int w1_layout(long long n, long long m, int K, W1Layout* L) {
    const long long terms = n + m - 1;
    L->tiles = terms > 0 ? (int)((terms + kW1Tile - 1) / kW1Tile) : 1;
    size_t tn = 0, tm = 0;
    cub::DoubleBuffer<uint32_t> none(nullptr, nullptr);
    if (n > 0)
        if (int rc = cuda_ok(cub::DeviceRadixSort::SortKeys(nullptr, tn, none, (int)n, 0, 32), "wasserstein1d sort size")) return rc;
    if (m > 0)
        if (int rc = cuda_ok(cub::DeviceRadixSort::SortKeys(nullptr, tm, none, (int)m, 0, 32), "wasserstein1d sort size")) return rc;
    const size_t keys = (size_t)K * (size_t)(n + m) * sizeof(uint32_t);
    L->counts = 0;
    L->keys_a = align256(2 * (size_t)K * sizeof(unsigned long long));
    L->keys_b = L->keys_a + align256(keys);
    L->partial = L->keys_b + align256(keys);
    L->temp = L->partial + align256((size_t)K * L->tiles * sizeof(double));
    L->temp_bytes = tn > tm ? tn : tm;
    L->total = L->temp + align256(L->temp_bytes > 0 ? L->temp_bytes : 1);
    return MMB_OK;
}

// sorts the K columns of one sample in place; returns in *sorted the buffer (keys_a or keys_b) that holds them
int w1_sort(uint32_t* ka, uint32_t* kb, long long rows, int K, void* temp, size_t temp_bytes, uint32_t** sorted, cudaStream_t stream) {
    *sorted = ka;
    if (rows == 0) return MMB_OK;
    int selector = 0;
    for (int c = 0; c < K; ++c) {
        cub::DoubleBuffer<uint32_t> db(ka + c * rows, kb + c * rows);
        size_t tb = temp_bytes;
        if (int rc = cuda_ok(cub::DeviceRadixSort::SortKeys(temp, tb, db, (int)rows, 0, 32, stream), "wasserstein1d sort")) return rc;
        selector = db.selector;   // set on the host from the number of passes, which depends only on rows: the same for every column
    }
    *sorted = selector ? kb : ka;
    return MMB_OK;
}

}  // namespace

size_t wasserstein1d_workspace_bytes(int n, int m, int K) {
    W1Layout L;
    return w1_layout(n, m, K, &L) == MMB_OK ? L.total : 0;
}

int launch_wasserstein1d(const float* x, long long ldx, int n, const float* y, long long ldy, int m, int K, double* out, long long* n_used,
                         void* workspace, cudaStream_t stream) {
    W1Layout L;
    if (int rc = w1_layout(n, m, K, &L)) return rc;
    char* ws = static_cast<char*>(workspace);
    auto* finite = reinterpret_cast<unsigned long long*>(ws + L.counts);
    auto* ka = reinterpret_cast<uint32_t*>(ws + L.keys_a);
    auto* kb = reinterpret_cast<uint32_t*>(ws + L.keys_b);
    auto* partial = reinterpret_cast<double*>(ws + L.partial);
    void* temp = ws + L.temp;
    const long long xo = (long long)K * n;   // y's keys follow x's
    if (int rc = cuda_ok(cudaMemsetAsync(finite, 0, 2 * (size_t)K * sizeof(unsigned long long), stream), "wasserstein1d counts")) return rc;
    auto key_blocks = [K](long long rows) {
        const long long b = (rows * K + kW1Threads - 1) / kW1Threads;
        return (int)(b < kKeyBlocks ? b : kKeyBlocks);
    };
    if (n > 0) w1_keys_kernel<<<key_blocks(n), kW1Threads, 0, stream>>>(x, ldx, n, K, ka, finite);
    if (m > 0) w1_keys_kernel<<<key_blocks(m), kW1Threads, 0, stream>>>(y, ldy, m, K, ka + xo, finite + K);
    if (int rc = cuda_ok(cudaGetLastError(), "w1_keys launch")) return rc;
    uint32_t *xs, *ys;
    if (int rc = w1_sort(ka, kb, n, K, temp, L.temp_bytes, &xs, stream)) return rc;
    if (int rc = w1_sort(ka + xo, kb + xo, m, K, temp, L.temp_bytes, &ys, stream)) return rc;
    w1_merge_kernel<<<dim3(L.tiles, K), kW1Threads, 0, stream>>>(xs, n, ys, m, finite, K, partial);
    w1_final_kernel<<<1, kW1Threads, 0, stream>>>(partial, L.tiles, finite, K, out, n_used);
    return cuda_ok(cudaGetLastError(), "wasserstein1d launch");
}

}  // namespace mmb
