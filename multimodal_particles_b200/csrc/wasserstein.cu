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
//
// launch_wasserstein1d_drawn computes the same quantity per draw t and feature c over the used slots of drawn jets
// (JetNet's W1-P / W1-M / W1-EFP draws), without materialising the drawn samples and without a host synchronisation:
//   1. w1_drawn_count_kernel counts the used slots of every drawn jet; one CUB inclusive scan over all draws of both samples
//      gives each drawn jet its offset in its draw's sample and each draw its length (integers: exact).
//   2. w1_drawn_keys_kernel writes the keys of the used slots into one segment per (sample, draw, feature), each of the
//      host-known capacity rows * P; the tail of a segment keeps the kNoKey fill, so it sorts last and is never read.
//   3. w1_sort sorts every segment over its full capacity (one CUB radix sort each; the host-known length is what lets the
//      sorts be launched without reading a length back).
//   4. w1_drawn_merge_kernel / w1_drawn_final_kernel run w1_merge_terms and w1_column per segment with the tile count
//      w1_tiles(n_t, m_t) of the draw's own lengths (grids are sized for the capacity; tiles past the end exit), so every
//      value is bit-identical to launch_wasserstein1d on the materialised draw.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

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

// tiles of the merged sequence of n and m rows (a compile-time tile, so the fixed-shape sums below depend only on the rows)
__host__ __device__ __forceinline__ long long w1_tiles(long long n, long long m) {
    const long long terms = n + m - 1;
    return terms > 0 ? (terms + kW1Tile - 1) / kW1Tile : 1;
}

// this thread's share of tile `tile`: the sum over its kW1Items terms k of |i_k m' - j_k n'| (z_{k+1} - z_k), k < n' + m' - 1,
// of the merge of the sorted finite keys a[0..nx) and b[0..ny)
__device__ __forceinline__ double w1_merge_terms(const uint32_t* __restrict__ a, long long nx, const uint32_t* __restrict__ b,
                                                 long long ny, long long tile) {
    const long long terms = nx + ny - 1;
    const long long k0 = tile * kW1Tile + (long long)threadIdx.x * kW1Items;
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
    return s;
}

// one block: the partials p[0..tiles) of one column in a fixed order (thread t adds its run of `per`, then the tree) / (n' m'),
// NaN when a sample has no finite value
__device__ __forceinline__ double w1_column(const double* __restrict__ p, long long tiles, unsigned long long nx, unsigned long long ny,
                                           double* red) {
    const long long per = (tiles + kW1Threads - 1) / kW1Threads;
    double s = 0.0;
    for (long long t = threadIdx.x * per, t1 = min(t + per, tiles); t < t1; ++t) s += p[t];
    const double total = block_sum(s, red);
    return (nx && ny) ? total / ((double)nx * (double)ny) : __longlong_as_double(0x7FF8000000000000LL);
}

// grid (tiles, K): partial[c][tile] = the block's sum of w1_merge_terms
__global__ void __launch_bounds__(kW1Threads) w1_merge_kernel(const uint32_t* __restrict__ xs, long long n, const uint32_t* __restrict__ ys,
                                                              long long m, const unsigned long long* __restrict__ finite, int K,
                                                              double* __restrict__ partial) {
    __shared__ double red[kW1Threads];
    const int c = blockIdx.y;
    const long long nx = (long long)finite[c], ny = (long long)finite[K + c];
    const double t = block_sum(w1_merge_terms(xs + c * n, nx, ys + c * m, ny, blockIdx.x), red);
    if (threadIdx.x == 0) partial[c * (long long)gridDim.x + blockIdx.x] = t;
}

// one block: out[c] = w1_column of column c
__global__ void __launch_bounds__(kW1Threads) w1_final_kernel(const double* __restrict__ partial, int tiles,
                                                              const unsigned long long* __restrict__ finite, int K,
                                                              double* __restrict__ out, long long* __restrict__ n_used) {
    __shared__ double red[kW1Threads];
    for (int c = 0; c < K; ++c) {
        const unsigned long long nx = finite[c], ny = finite[K + c];
        const double w = w1_column(partial + (long long)c * tiles, tiles, nx, ny, red);
        if (threadIdx.x == 0) {
            out[c] = w;
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
    L->tiles = (int)w1_tiles(n, m);
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

namespace {
// ---- drawn samples -----------------------------------------------------------------------------------------------------------

constexpr int kDrawnWarps = kW1Threads / 32;

struct DrawnSample {   // jet j, slot p, feature c at v[j*ld_jet + p*ld_slot + c]; used iff !mask || mask[j*ldm + p]
    const float* v;
    long long ld_jet, ld_slot;
    const uint8_t* mask;
    long long ldm;
    const int32_t* idx;   // [draws][rows]
};

__device__ __forceinline__ bool drawn_used(const DrawnSample& S, long long j, int p) { return !S.mask || S.mask[j * S.ldm + p] != 0; }

// start of the sample of (side, draw) q = side * draws + t in the drawn-jet order, from the inclusive scan of the jet counts
__device__ __forceinline__ long long drawn_base(const long long* __restrict__ inc, long long q, long long rows) {
    return q == 0 ? 0 : inc[q * rows - 1];
}
__device__ __forceinline__ long long drawn_len(const long long* __restrict__ inc, long long q, long long rows) {
    return inc[(q + 1) * rows - 1] - drawn_base(inc, q, rows);
}

// one warp per drawn jet e of [2][draws][rows]: cnt[e] = its used slots
__global__ void __launch_bounds__(kW1Threads) w1_drawn_count_kernel(DrawnSample x, DrawnSample y, int P, long long jets,
                                                                    long long* __restrict__ cnt) {
    const long long e = blockIdx.x * (long long)kDrawnWarps + (threadIdx.x >> 5);
    if (e >= 2 * jets) return;
    const DrawnSample& S = e < jets ? x : y;
    const long long j = S.idx[e < jets ? e : e - jets];
    int used = 0;
    for (int p0 = 0; p0 < P; p0 += 32) {
        const int p = p0 + (threadIdx.x & 31);
        used += __popc(__ballot_sync(0xFFFFFFFFu, p < P && drawn_used(S, j, p)));
    }
    if ((threadIdx.x & 31) == 0) cnt[e] = used;
}

// grid (ceil(rows / kDrawnWarps), <= 2 draws): one warp per drawn jet writes the keys of its used slots, in slot order, at its
// offset of the segments (q, c); finite[q][c] += finite values
__global__ void __launch_bounds__(kW1Threads) w1_drawn_keys_kernel(DrawnSample x, DrawnSample y, int P, int F, int draws, long long rows,
                                                                   long long cap, const long long* __restrict__ cnt,
                                                                   const long long* __restrict__ inc, uint32_t* __restrict__ keys,
                                                                   unsigned long long* __restrict__ finite) {
    __shared__ unsigned int fin[MMB_W1_MAX_K];
    const int lane = threadIdx.x & 31;
    const long long r = blockIdx.x * (long long)kDrawnWarps + (threadIdx.x >> 5);
    for (long long q = blockIdx.y; q < 2LL * draws; q += gridDim.y) {
        for (int c = threadIdx.x; c < F; c += blockDim.x) fin[c] = 0;
        __syncthreads();
        if (r < rows) {
            const DrawnSample& S = q < draws ? x : y;
            const long long e = q * rows + r;
            const long long j = S.idx[e - (q < draws ? 0 : draws * rows)];
            long long pos = inc[e] - cnt[e] - drawn_base(inc, q, rows);
            uint32_t* seg = keys + q * F * cap;
            for (int p0 = 0; p0 < P; p0 += 32) {
                const int p = p0 + lane;
                const bool used = p < P && drawn_used(S, j, p);
                const unsigned bal = __ballot_sync(0xFFFFFFFFu, used);
                if (used) {
                    const long long at = pos + __popc(bal & ((1u << lane) - 1u));
                    const float* v = S.v + j * S.ld_jet + (long long)p * S.ld_slot;
                    for (int c = 0; c < F; ++c) {
                        const uint32_t key = w1_key(v[c]);
                        seg[c * cap + at] = key;
                        if (key != kNoKey) atomicAdd(&fin[c], 1u);
                    }
                }
                pos += __popc(bal);
            }
        }
        __syncthreads();
        for (int c = threadIdx.x; c < F; c += blockDim.x)
            if (fin[c]) atomicAdd(&finite[q * F + c], (unsigned long long)fin[c]);
        __syncthreads();
    }
}

// grid (tiles of the capacity, <= draws * F): partial[t*F + c][tile] = the block's sum of w1_merge_terms over the draw's tiles
__global__ void __launch_bounds__(kW1Threads) w1_drawn_merge_kernel(const uint32_t* __restrict__ sorted, long long cap, int F, int draws,
                                                                    long long rows, const long long* __restrict__ inc,
                                                                    const unsigned long long* __restrict__ finite, long long tiles_cap,
                                                                    double* __restrict__ partial) {
    __shared__ double red[kW1Threads];
    const long long segs = (long long)draws * F;
    for (long long g = blockIdx.y; g < segs; g += gridDim.y) {
        const long long t = g / F;
        if ((long long)blockIdx.x >= w1_tiles(drawn_len(inc, t, rows), drawn_len(inc, draws + t, rows))) continue;   // block-uniform
        const long long nx = (long long)finite[g], ny = (long long)finite[segs + g];
        const double s = block_sum(w1_merge_terms(sorted + g * cap, nx, sorted + (segs + g) * cap, ny, blockIdx.x), red);
        if (threadIdx.x == 0) partial[g * tiles_cap + blockIdx.x] = s;
    }
}

// grid (<= draws * F): out[t*F + c] = w1_column of the draw's tiles; n_used [2][draws][F]
__global__ void __launch_bounds__(kW1Threads) w1_drawn_final_kernel(const double* __restrict__ partial, long long tiles_cap, int F,
                                                                    int draws, long long rows, const long long* __restrict__ inc,
                                                                    const unsigned long long* __restrict__ finite, double* __restrict__ out,
                                                                    long long* __restrict__ n_used) {
    __shared__ double red[kW1Threads];
    const long long segs = (long long)draws * F;
    for (long long g = blockIdx.x; g < segs; g += gridDim.x) {
        const long long t = g / F;
        const unsigned long long nx = finite[g], ny = finite[segs + g];
        const double w = w1_column(partial + g * tiles_cap, w1_tiles(drawn_len(inc, t, rows), drawn_len(inc, draws + t, rows)), nx, ny, red);
        if (threadIdx.x == 0) {
            out[g] = w;
            if (n_used) {
                n_used[g] = (long long)nx;
                n_used[segs + g] = (long long)ny;
            }
        }
    }
}

struct DrawnLayout {
    size_t finite, cnt, inc, keys_a, keys_b, partial, temp, temp_bytes, total;
    long long cap, tiles_cap;
};

// workspace: finite counts [2][draws][F] u64 | jet counts [2][draws][rows] i64 | their inclusive scan | keys [2][draws][F][cap] u32
// | alternate keys | partials [draws][F][tiles_cap] f64 | CUB temp (scan or sort)
int drawn_layout(int draws, int rows, int P, int F, DrawnLayout* L) {
    L->cap = (long long)rows * P;
    L->tiles_cap = w1_tiles(L->cap, L->cap);
    const long long jets = 2LL * draws * rows;
    size_t ts = 0, tk = 0;
    if (int rc = cuda_ok(cub::DeviceScan::InclusiveSum(nullptr, ts, (const long long*)nullptr, (long long*)nullptr, jets),
                         "wasserstein1d_drawn scan size"))
        return rc;
    cub::DoubleBuffer<uint32_t> none(nullptr, nullptr);
    if (int rc = cuda_ok(cub::DeviceRadixSort::SortKeys(nullptr, tk, none, (int)L->cap, 0, 32), "wasserstein1d_drawn sort size")) return rc;
    const size_t keys = 2 * (size_t)draws * F * (size_t)L->cap * sizeof(uint32_t);
    L->finite = 0;
    L->cnt = align256(2 * (size_t)draws * F * sizeof(unsigned long long));
    L->inc = L->cnt + align256((size_t)jets * sizeof(long long));
    L->keys_a = L->inc + align256((size_t)jets * sizeof(long long));
    L->keys_b = L->keys_a + align256(keys);
    L->partial = L->keys_b + align256(keys);
    L->temp = L->partial + align256((size_t)draws * F * (size_t)L->tiles_cap * sizeof(double));
    L->temp_bytes = ts > tk ? ts : tk;
    L->total = L->temp + align256(L->temp_bytes > 0 ? L->temp_bytes : 1);
    return MMB_OK;
}

}  // namespace

size_t wasserstein1d_drawn_workspace_bytes(int draws, int rows, int P, int F) {
    DrawnLayout L;
    return drawn_layout(draws, rows, P, F, &L) == MMB_OK ? L.total : 0;
}

int launch_wasserstein1d_drawn(const float* x, long long ldx_jet, long long ldx_slot, const uint8_t* mask_x, long long ldmx, const float* y,
                               long long ldy_jet, long long ldy_slot, const uint8_t* mask_y, long long ldmy, int P, int F, const int32_t* idx_x,
                               const int32_t* idx_y, int draws, int rows, double* out, long long* n_used, void* workspace,
                               cudaStream_t stream) {
    DrawnLayout L;
    if (int rc = drawn_layout(draws, rows, P, F, &L)) return rc;
    char* ws = static_cast<char*>(workspace);
    auto* finite = reinterpret_cast<unsigned long long*>(ws + L.finite);
    auto* cnt = reinterpret_cast<long long*>(ws + L.cnt);
    auto* inc = reinterpret_cast<long long*>(ws + L.inc);
    auto* ka = reinterpret_cast<uint32_t*>(ws + L.keys_a);
    auto* kb = reinterpret_cast<uint32_t*>(ws + L.keys_b);
    auto* partial = reinterpret_cast<double*>(ws + L.partial);
    const DrawnSample sx{x, ldx_jet, ldx_slot, mask_x, ldmx, idx_x}, sy{y, ldy_jet, ldy_slot, mask_y, ldmy, idx_y};
    const long long jets = (long long)draws * rows;
    const int segs = 2 * draws * F;
    auto grid_y = [](long long v) { return (unsigned)(v < 65535 ? v : 65535); };
    if (int rc = cuda_ok(cudaMemsetAsync(finite, 0, (size_t)segs * sizeof(unsigned long long), stream), "wasserstein1d_drawn counts")) return rc;
    if (int rc = cuda_ok(cudaMemsetAsync(ka, 0xFF, (size_t)segs * L.cap * sizeof(uint32_t), stream), "wasserstein1d_drawn fill")) return rc;
    w1_drawn_count_kernel<<<(unsigned)((2 * jets + kDrawnWarps - 1) / kDrawnWarps), kW1Threads, 0, stream>>>(sx, sy, P, jets, cnt);
    if (int rc = cuda_ok(cudaGetLastError(), "w1_drawn_count launch")) return rc;
    size_t tb = L.temp_bytes;
    if (int rc = cuda_ok(cub::DeviceScan::InclusiveSum(ws + L.temp, tb, (const long long*)cnt, inc, 2 * jets, stream), "wasserstein1d_drawn scan"))
        return rc;
    w1_drawn_keys_kernel<<<dim3((unsigned)((rows + kDrawnWarps - 1) / kDrawnWarps), grid_y(2LL * draws)), kW1Threads, 0, stream>>>(
        sx, sy, P, F, draws, rows, L.cap, cnt, inc, ka, finite);
    if (int rc = cuda_ok(cudaGetLastError(), "w1_drawn_keys launch")) return rc;
    uint32_t* sorted;
    if (int rc = w1_sort(ka, kb, L.cap, segs, ws + L.temp, L.temp_bytes, &sorted, stream)) return rc;
    w1_drawn_merge_kernel<<<dim3((unsigned)L.tiles_cap, grid_y((long long)draws * F)), kW1Threads, 0, stream>>>(
        sorted, L.cap, F, draws, rows, inc, finite, L.tiles_cap, partial);
    w1_drawn_final_kernel<<<grid_y((long long)draws * F), kW1Threads, 0, stream>>>(partial, L.tiles_cap, F, draws, rows, inc, finite, out,
                                                                                     n_used);
    return cuda_ok(cudaGetLastError(), "wasserstein1d_drawn launch");
}

}  // namespace mmb
