// w1_sort_choice.cu — the sort stage of mmb_wasserstein1d_drawn (DESIGN.md §4.6e) at JetNet's W1-P defaults, four ways.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o w1_sort_choice w1_sort_choice.cu && ./w1_sort_choice
// 30 segments (2 samples x 5 draws x 3 features) of capacity rows * P = 50 000 * 128 keys, the used length of each known only on
// the device; the tail of a segment holds 0xFFFFFFFF.  Lengths: JetClass-like (about 35 % of the capacity) or full.
//   per_segment    one cub::DeviceRadixSort per segment over its whole capacity (what the library does);
//   segmented      cub::DeviceSegmentedSort over [seg * cap, seg * cap + len) with device-side offsets;
//   segmented_rdx  cub::DeviceSegmentedRadixSort over the same device-side ranges;
//   key64          one cub::DeviceRadixSort of (segment << 32 | key) over every capacity, 37 bits.
// Device time by CUDA events around --reps sorts, each after a device-to-device copy of the unsorted keys; the copies alone
// are timed the same way and subtracted.  Every variant's sorted used prefixes are compared with per_segment's.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <functional>
#include <vector>

#define CK(x)                                                                                  \
    do {                                                                                       \
        cudaError_t e_ = (x);                                                                  \
        if (e_ != cudaSuccess) {                                                               \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
            exit(1);                                                                           \
        }                                                                                      \
    } while (0)

static const int kSegs = 30, kReps = 10;
static const long long kCap = 50000LL * 128;

__global__ void fill_keys(uint32_t* k, const long long* len, long long cap, uint64_t seed) {
    const long long seg = blockIdx.y;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < cap; i += (long long)gridDim.x * blockDim.x) {
        uint64_t z = (seed + seg * cap + i) * 0x9E3779B97F4A7C15ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        k[seg * cap + i] = i < len[seg] ? (uint32_t)(z >> 33) | 0x80000000u : 0xFFFFFFFFu;   // positive-float-like keys
    }
}

__global__ void to_key64(const uint32_t* k, uint64_t* k64, long long cap) {
    const long long seg = blockIdx.y;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < cap; i += (long long)gridDim.x * blockDim.x)
        k64[seg * cap + i] = ((uint64_t)seg << 32) | k[seg * cap + i];
}

__global__ void low_half(const uint64_t* k64, uint32_t* k, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) k[i] = (uint32_t)k64[i];
}

__global__ void offsets(const long long* len, long long cap, long long* begin, long long* end) {
    const int s = threadIdx.x;
    if (s < kSegs) {
        begin[s] = s * cap;
        end[s] = s * cap + len[s];
    }
}

template <class F>
static float timed(F&& body, cudaEvent_t a, cudaEvent_t b) {
    body();   // warm-up
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    for (int r = 0; r < kReps; ++r) body();
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms;
    CK(cudaEventElapsedTime(&ms, a, b));
    return ms / kReps;
}

int main() {
    const long long total = kSegs * kCap;
    uint32_t *src, *ka, *kb;
    uint64_t *k64a, *k64b;
    long long *len, *begin, *end;
    CK(cudaMalloc(&src, total * 4));
    CK(cudaMalloc(&ka, total * 4));
    CK(cudaMalloc(&kb, total * 4));
    CK(cudaMalloc(&k64a, total * 8));
    CK(cudaMalloc(&k64b, total * 8));
    CK(cudaMalloc(&len, kSegs * 8));
    CK(cudaMalloc(&begin, kSegs * 8));
    CK(cudaMalloc(&end, kSegs * 8));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    std::vector<uint32_t> ref(total), got(total);
    printf("{\"measure\": \"w1_drawn_sort_choice\", \"segments\": %d, \"capacity\": %lld, \"reps\": %d, \"rows\": [", kSegs, kCap, kReps);
    for (int full = 0; full < 2; ++full) {
        std::vector<long long> hl(kSegs);
        srand(1);
        for (int s = 0; s < kSegs; ++s) hl[s] = full ? kCap : (long long)(kCap * (0.35 + 0.01 * (rand() % 5 - 2)));
        CK(cudaMemcpy(len, hl.data(), kSegs * 8, cudaMemcpyHostToDevice));
        fill_keys<<<dim3(1024, kSegs), 256>>>(src, len, kCap, 12345);
        offsets<<<1, 32>>>(len, kCap, begin, end);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
        size_t t1 = 0, t2 = 0, t3 = 0, t4 = 0;
        cub::DoubleBuffer<uint32_t> none(nullptr, nullptr);
        cub::DoubleBuffer<uint64_t> none64(nullptr, nullptr);
        CK(cub::DeviceRadixSort::SortKeys(nullptr, t1, none, (int)kCap, 0, 32));
        CK(cub::DeviceSegmentedSort::SortKeys(nullptr, t2, none, total, kSegs, begin, end));
        CK(cub::DeviceSegmentedRadixSort::SortKeys(nullptr, t3, none, total, kSegs, begin, end, 0, 32));
        CK(cub::DeviceRadixSort::SortKeys(nullptr, t4, none64, total, 0, 37));
        size_t tb = t1 > t2 ? t1 : t2;
        tb = tb > t3 ? tb : t3;
        tb = tb > t4 ? tb : t4;
        void* temp;
        CK(cudaMalloc(&temp, tb));
        auto copy = [&] { CK(cudaMemcpyAsync(ka, src, total * 4, cudaMemcpyDeviceToDevice)); };
        const float copy_ms = timed(copy, a, b);
        uint32_t* out = nullptr;
        auto per_segment = [&] {
            copy();
            int sel = 0;
            for (int s = 0; s < kSegs; ++s) {
                cub::DoubleBuffer<uint32_t> db(ka + s * kCap, kb + s * kCap);
                size_t t = tb;
                CK(cub::DeviceRadixSort::SortKeys(temp, t, db, (int)kCap, 0, 32));
                sel = db.selector;
            }
            out = sel ? kb : ka;
        };
        auto segmented = [&] {
            copy();
            cub::DoubleBuffer<uint32_t> db(ka, kb);
            size_t t = tb;
            CK(cub::DeviceSegmentedSort::SortKeys(temp, t, db, total, kSegs, begin, end));
            out = db.Current();
        };
        auto segmented_rdx = [&] {
            copy();
            cub::DoubleBuffer<uint32_t> db(ka, kb);
            size_t t = tb;
            CK(cub::DeviceSegmentedRadixSort::SortKeys(temp, t, db, total, kSegs, begin, end, 0, 32));
            out = db.Current();
        };
        auto key64 = [&] {
            copy();
            to_key64<<<dim3(1024, kSegs), 256>>>(ka, k64a, kCap);
            cub::DoubleBuffer<uint64_t> db(k64a, k64b);
            size_t t = tb;
            CK(cub::DeviceRadixSort::SortKeys(temp, t, db, total, 0, 37));
            low_half<<<4096, 256>>>(db.Current(), kb, total);
            out = kb;
        };
        const char* names[4] = {"per_segment", "segmented", "segmented_rdx", "key64"};
        float ms[4];
        ms[0] = timed(per_segment, a, b) - copy_ms;
        CK(cudaMemcpy(ref.data(), out, total * 4, cudaMemcpyDeviceToHost));
        bool same[4] = {true, true, true, true};
        for (int v = 1; v < 4; ++v) {
            ms[v] = timed(v == 1 ? std::function<void()>(segmented) : v == 2 ? std::function<void()>(segmented_rdx) : std::function<void()>(key64), a, b) -
                    copy_ms;
            CK(cudaMemcpy(got.data(), out, total * 4, cudaMemcpyDeviceToHost));
            for (int s = 0; s < kSegs; ++s)
                same[v] = same[v] && memcmp(ref.data() + s * kCap, got.data() + s * kCap, hl[s] * 4) == 0;
        }
        printf("%s{\"lengths\": \"%s\", \"used_keys\": %lld, \"copy_ms\": %.4f", full ? ", " : "", full ? "full" : "about 35 % of capacity",
               [&] { long long u = 0; for (long long l : hl) u += l; return u; }(), copy_ms);
        for (int v = 0; v < 4; ++v) printf(", \"%s_ms\": %.4f, \"%s_same_prefixes\": %s", names[v], ms[v], names[v], same[v] ? "true" : "false");
        printf("}");
        CK(cudaFree(temp));
    }
    printf("]}\n");
    return 0;
}
